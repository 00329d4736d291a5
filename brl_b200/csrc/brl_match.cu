// brl_match.cu -- a whole duplicate match as one stream-ordered call (brl_duplicate_match): make_simple_duplicate_evaluate
// (src/evaluation.py:69-204) for every env of the batch, its `lax.while_loop` (:120-171) run on the device by a CUDA graph
// WHILE node.  sm_100a only.
//
//   init (brl_init) -> Table_info A / B (brl_state_fields) -> grouping (brl_model_rows) -> control
//   WHILE (control said so) {
//       [path kernel -> IF fused forward / IF per-layer forward]    the grouped forward, sized from the device count
//       brl_duplicate_step -> cum_return += rewards[:, 0] -> grouping -> control
//   }
//   match sums (brl_match_stats_ranges, or brl_match_stats for one range)
//
// The control kernel reads the padded row count brl_model_rows left in offsets[M] and sets the loop's condition: the loop
// ends when no env is live, when a live env's net id is outside [0, M), or at BRL_MATCH_MAX_STEPS forwards; the last two
// write a status.  Nothing is read back to the host.  The forward path follows the host's rule (fused from kPairMinM rows
// on, per-layer below, unless BRL_F_TUNE_MLP_LAYERS / BRL_F_TUNE_MLP_FUSED pin it), applied to the device count by a
// path kernel and two IF nodes.
//
// On a plain stream the graph is captured on a private stream, instantiated once per set of buffers and parameters
// (cached), and launched.  On a stream that is being captured (torch.cuda.graph, an XLA command buffer) the same nodes
// go into the caller's capture.
#include <cstring>
#include <map>
#include <mutex>
#include <string>

#include "common.h"

namespace brl {

int32_t launch_policy_grouped_dev(cudaStream_t s, int32_t flags, int64_t capacity, int n_models, const void* obs,
                                  const unsigned char* pool, unsigned char* scratch, const uint8_t* mask, int32_t* action,
                                  const int32_t* rows, const int32_t* block_model, const int32_t* n_rows);
int32_t warm_policy_grouped_dev(bool split);

// ---- kernels -----------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pair_models(int32_t* __restrict__ env_models, int64_t n) {  // every env: net 0 vs net 1
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) reinterpret_cast<int2*>(env_models)[i] = make_int2(0, 1);
}

__global__ void __launch_bounds__(256) k_add_reward(float* __restrict__ cum_return, const float4* __restrict__ rewards, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) cum_return[i] += rewards[i].x;  // cum_return += state.rewards[:, 0] (src/evaluation.py:167-169)
}

// after each grouping: continue while rows are live; stop with a status on a bad net id or at the step bound.  `iter` counts
// the forwards the loop has been allowed to run.
__global__ void k_match_control(const int32_t* __restrict__ n_rows, int32_t* __restrict__ iter, int32_t* __restrict__ status,
                                cudaGraphConditionalHandle loop) {
    const int rows = *n_rows, it = *iter;
    bool go = rows > 0;
    if (rows < 0) {
        *status = BRL_MATCH_BAD_MODEL;
    } else if (go && it >= BRL_MATCH_MAX_STEPS) {
        *status = BRL_MATCH_STEP_BOUND;
        go = false;
    }
    if (go) *iter = it + 1;
    cudaGraphSetConditional(loop, go ? 1u : 0u);
}

// the forward's path for this iteration's count: fused_forward() of brl_mlp.cu on the device
__global__ void k_match_path(const int32_t* __restrict__ n_rows, cudaGraphConditionalHandle fused, cudaGraphConditionalHandle layers) {
    const bool f = *n_rows >= kPairMinM;
    cudaGraphSetConditional(fused, f ? 1u : 0u);
    cudaGraphSetConditional(layers, f ? 0u : 1u);
}

// ---- the scratch ----------------------------------------------------------------------------------------------------------
struct MatchLayout {
    size_t state, obs, mask, rewards, terminated, player, action, info[2][6], env_models, rows, counts, offsets, block_model, ctl,
        forward, total;
};

static MatchLayout match_layout(int64_t n, int64_t M) {
    MatchLayout L{};
    size_t off = 0;
    auto take = [&](size_t bytes) {
        const size_t at = off;
        off = (off + bytes + 255) & ~(size_t)255;
        return at;
    };
    const size_t un = (size_t)n, cap = (size_t)brl_model_rows_capacity(n, M);
    L.state = take(BRL_STATE_PLANES * 16 * un);
    L.obs = take(un * BRL_OBS_DIM * 2);
    L.mask = take(un * BRL_NUM_ACTIONS);
    L.rewards = take(un * 16);
    L.terminated = take(un);
    L.player = take(un);
    L.action = take(un * 4);
    for (int t = 0; t < 2; ++t) {  // Table_info: terminated, rewards[4], last_bid, last_bidder, call_x, call_xx
        L.info[t][0] = take(un);
        L.info[t][1] = take(un * 16);
        L.info[t][2] = take(un * 4);
        L.info[t][3] = take(un * 4);
        L.info[t][4] = take(un);
        L.info[t][5] = take(un);
    }
    L.env_models = take(un * 8);
    L.rows = take(cap * 4);
    L.counts = take((size_t)M * 4);
    L.offsets = take((size_t)(M + 1) * 4);
    L.block_model = take(cap / kGroupRows * 4);
    L.ctl = take(16);  // i32 iteration counter
    L.forward = take((size_t)brl_policy_grouped_scratch_bytes(n, M));
    L.total = off;
    return L;
}

// every device pointer and size one match needs
struct MatchPlan {
    int64_t n, cap, P;
    int M;
    int32_t n_deals, flags;
    float illegal_penalty, illegal_bonus;
    const void *keys, *table;
    const unsigned char* pool;
    const int64_t* ranges;
    float* cum_return;
    double* sums;
    int32_t* status;
    void* info[2][6];
    unsigned char* scratch;
    MatchLayout L;
    int32_t* env_models;  // the caller's, or (NULL given) the scratch's, filled with net 0 vs net 1
    bool default_models;
    template <class T = void>
    T* at(size_t off) const { return reinterpret_cast<T*>(scratch + off); }
    int32_t* offsets() const { return at<int32_t>(L.offsets); }
};

static BrlParams env_params(const MatchPlan& q, int64_t n) {
    BrlParams p{};
    p.n_envs = n;
    p.state_stride = q.n;
    p.n_deals = q.n_deals;
    p.flags = BRL_F_OBS_BF16;
    p.illegal_penalty = q.illegal_penalty;
    p.illegal_bonus = q.illegal_bonus;
    return p;
}

// a failed graph-building call: its CUDA error, or a plain failure when the call left none
static int32_t launch_error(const char* what) {
    const int32_t rc = check_launch(what);
    return rc != BRL_OK ? rc : fail(BRL_E_LAUNCH, "%s failed", what);
}

static int32_t model_rows(const MatchPlan& q, cudaStream_t s) {
    void* b[7] = {q.at(q.L.player), q.at(q.L.terminated), q.env_models, q.at(q.L.rows), q.at(q.L.counts), q.offsets(),
                  q.at(q.L.block_model)};
    BrlParams p = env_params(q, q.n);
    p.k_steps = q.M;
    return brl_model_rows(s, b, &p, sizeof(p));
}

static int32_t control(const MatchPlan& q, cudaStream_t s, cudaGraphConditionalHandle loop) {
    k_match_control<<<1, 1, 0, s>>>(q.offsets() + q.M, q.at<int32_t>(q.L.ctl), q.status, loop);
    return check_launch("brl_duplicate_match (control)");
}

// the capture's graph, with the stream's current dependencies; a conditional node of `type` there (its body in *body), made
// the stream's only dependency
static int32_t add_conditional(cudaStream_t s, cudaGraphConditionalHandle h, cudaGraphConditionalNodeType type, cudaGraph_t* body) {
    cudaStreamCaptureStatus st;
    cudaGraph_t g = nullptr;
    const cudaGraphNode_t* deps = nullptr;
    size_t n_deps = 0;
    if (cudaStreamGetCaptureInfo(s, &st, nullptr, &g, &deps, &n_deps) != cudaSuccess || st != cudaStreamCaptureStatusActive)
        return launch_error("brl_duplicate_match (capture info)");
    cudaGraphNodeParams cp{};
    cp.type = cudaGraphNodeTypeConditional;
    cp.conditional.handle = h;
    cp.conditional.type = type;
    cp.conditional.size = 1;
    cudaGraphNode_t node;
    if (cudaGraphAddNode(&node, g, deps, n_deps, &cp) != cudaSuccess ||
        cudaStreamUpdateCaptureDependencies(s, &node, 1, cudaStreamSetCaptureDependencies) != cudaSuccess)
        return launch_error("brl_duplicate_match (conditional node)");
    *body = cp.conditional.phGraph_out[0];
    return BRL_OK;
}

static int32_t new_handle(cudaStream_t s, cudaGraphConditionalHandle* h) {
    cudaStreamCaptureStatus st;
    cudaGraph_t g = nullptr;
    if (cudaStreamGetCaptureInfo(s, &st, nullptr, &g) != cudaSuccess || st != cudaStreamCaptureStatusActive ||
        cudaGraphConditionalHandleCreate(h, g, 0, cudaGraphCondAssignDefault) != cudaSuccess)
        return launch_error("brl_duplicate_match (conditional handle)");
    return BRL_OK;
}

// fill `body` by capturing what `fn(side)` enqueues on the side stream
template <class F>
static int32_t capture_into(cudaGraph_t body, cudaStream_t side, F&& fn) {
    if (cudaStreamBeginCaptureToGraph(side, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed) != cudaSuccess)
        return launch_error("brl_duplicate_match (body capture)");
    const int32_t rc = fn(side);
    cudaGraph_t out = nullptr;
    const cudaError_t end = cudaStreamEndCapture(side, &out);
    if (rc != BRL_OK) return rc;
    if (end != cudaSuccess) return launch_error("brl_duplicate_match (body capture)");
    return BRL_OK;
}

static int32_t forward(const MatchPlan& q, cudaStream_t s, int32_t path_flag) {
    const int32_t flags = (q.flags & BRL_F_MLP_BF16) | path_flag;
    return launch_policy_grouped_dev(s, flags, q.cap, q.M, q.at(q.L.obs), q.pool, q.at<unsigned char>(q.L.forward),
                                     q.at<uint8_t>(q.L.mask), q.at<int32_t>(q.L.action), q.at<int32_t>(q.L.rows),
                                     q.at<int32_t>(q.L.block_model), q.offsets() + q.M);
}

// one iteration of the loop (src/evaluation.py:124-169), on the body's capture stream s1; s2 captures the IF bodies
static int32_t emit_body(const MatchPlan& q, cudaStream_t s1, cudaStream_t s2, cudaGraphConditionalHandle loop) {
    int32_t rc;
    if (q.flags & BRL_F_TUNE_MLP_LAYERS) {
        rc = forward(q, s1, BRL_F_TUNE_MLP_LAYERS);
    } else if (q.flags & BRL_F_TUNE_MLP_FUSED) {
        rc = forward(q, s1, BRL_F_TUNE_MLP_FUSED);
    } else {
        cudaGraphConditionalHandle h_fused, h_layers;
        if ((rc = new_handle(s1, &h_fused)) || (rc = new_handle(s1, &h_layers))) return rc;
        k_match_path<<<1, 1, 0, s1>>>(q.offsets() + q.M, h_fused, h_layers);
        if ((rc = check_launch("brl_duplicate_match (path)"))) return rc;
        cudaGraph_t body;
        if ((rc = add_conditional(s1, h_fused, cudaGraphCondTypeIf, &body)) ||
            (rc = capture_into(body, s2, [&](cudaStream_t s) { return forward(q, s, BRL_F_TUNE_MLP_FUSED); })) ||
            (rc = add_conditional(s1, h_layers, cudaGraphCondTypeIf, &body)) ||
            (rc = capture_into(body, s2, [&](cudaStream_t s) { return forward(q, s, BRL_F_TUNE_MLP_LAYERS); })))
            return rc;
    }
    if (rc != BRL_OK) return rc;
    void* b[21] = {q.at(q.L.state), q.at(q.L.action), const_cast<void*>(q.table)};
    for (int t = 0; t < 2; ++t)
        for (int k = 0; k < 6; ++k) b[3 + 6 * t + k] = q.info[t][k];
    b[15] = q.at(q.L.state);
    b[16] = q.at(q.L.obs);
    b[17] = q.at(q.L.mask);
    b[18] = q.at(q.L.rewards);
    b[19] = q.at(q.L.terminated);
    b[20] = q.at(q.L.player);
    const BrlParams p = env_params(q, q.n);
    if ((rc = brl_duplicate_step(s1, b, &p, sizeof(p)))) return rc;  // src/evaluation.py:164
    k_add_reward<<<(unsigned)((q.n + 255) / 256), 256, 0, s1>>>(q.cum_return, q.at<float4>(q.L.rewards), q.n);
    if ((rc = check_launch("brl_duplicate_match (cum_return)"))) return rc;
    if ((rc = model_rows(q, s1))) return rc;
    return control(q, s1, loop);
}

// the whole match on the capturing stream s0 (its own capture, or the caller's)
static int32_t emit_match(const MatchPlan& q, cudaStream_t s0, cudaStream_t s1, cudaStream_t s2) {
    int32_t rc;
    cudaGraphConditionalHandle loop;
    if ((rc = new_handle(s0, &loop))) return rc;
    const size_t un = (size_t)q.n;
    if (cudaMemsetAsync(q.status, 0, sizeof(int32_t), s0) != cudaSuccess ||
        cudaMemsetAsync(q.at(q.L.ctl), 0, sizeof(int32_t), s0) != cudaSuccess ||
        cudaMemsetAsync(q.cum_return, 0, un * sizeof(float), s0) != cudaSuccess ||
        cudaMemsetAsync(q.at(q.L.action), 0, un * sizeof(int32_t), s0) != cudaSuccess)  // finished envs keep a (no-op) Pass
        return check_launch("brl_duplicate_match (memset)");
    if (q.default_models) k_pair_models<<<(unsigned)((q.n + 255) / 256), 256, 0, s0>>>(q.env_models, q.n);
    // src/evaluation.py:93-95: the envs from the given keys, observation in bf16 (what the forward reads)
    void* bi[8] = {const_cast<void*>(q.keys), const_cast<void*>(q.table), q.at(q.L.state), q.at(q.L.obs), q.at(q.L.mask),
                   q.at(q.L.rewards), q.at(q.L.terminated), q.at(q.L.player)};
    BrlParams p = env_params(q, q.n);
    if ((rc = brl_init(s0, bi, &p, sizeof(p)))) return rc;
    // :97-112 Table_info A = B = the init state's terminated, rewards, last_bid, last_bidder, call_x, call_xx
    void* bf[12] = {q.at(q.L.state), nullptr, nullptr, nullptr, nullptr, q.info[0][2], q.info[0][3], q.info[0][4], q.info[0][5]};
    if ((rc = brl_state_fields(s0, bf, &p, sizeof(p)))) return rc;
    const size_t bytes[6] = {un, un * 16, un * 4, un * 4, un, un};
    if (cudaMemcpyAsync(q.info[0][0], q.at(q.L.terminated), bytes[0], cudaMemcpyDeviceToDevice, s0) != cudaSuccess ||
        cudaMemcpyAsync(q.info[0][1], q.at(q.L.rewards), bytes[1], cudaMemcpyDeviceToDevice, s0) != cudaSuccess)
        return check_launch("brl_duplicate_match (Table_info)");
    for (int k = 0; k < 6; ++k)
        if (cudaMemcpyAsync(q.info[1][k], q.info[0][k], bytes[k], cudaMemcpyDeviceToDevice, s0) != cudaSuccess)
            return check_launch("brl_duplicate_match (Table_info)");
    if ((rc = model_rows(q, s0)) || (rc = control(q, s0, loop))) return rc;
    cudaGraph_t body;
    if ((rc = add_conditional(s0, loop, cudaGraphCondTypeWhile, &body)) ||
        (rc = capture_into(body, s1, [&](cudaStream_t s) { return emit_body(q, s, s2, loop); })))
        return rc;
    // :199-201 the match sums, per range
    if (q.ranges) {
        void* bs[3] = {q.cum_return, const_cast<int64_t*>(q.ranges), q.sums};
        BrlParams ps{};
        ps.n_envs = q.P;
        return brl_match_stats_ranges(s0, bs, &ps, sizeof(ps));
    }
    void* bs[2] = {q.cum_return, q.sums};
    BrlParams ps{};
    ps.n_envs = q.n;
    return brl_match_stats(s0, bs, &ps, sizeof(ps));
}

// ---- graph cache and capture streams ------------------------------------------------------------------------------------
struct MatchCache {
    std::mutex mu;
    std::map<std::string, std::pair<cudaGraphExec_t, uint64_t>> exec;  // key -> (instantiated graph, last use)
    cudaStream_t streams[kMaxDevices][3] = {};
    uint64_t clock = 0;
    long long builds = 0;
};
static MatchCache& cache() {
    static MatchCache* c = new MatchCache();  // never destroyed: instantiated graphs outlive static destruction order
    return *c;
}
constexpr size_t kMaxCachedGraphs = 16;

static int32_t capture_streams(cudaStream_t** out) {
    cudaStream_t* s = cache().streams[device_slot()];
    for (int k = 0; k < 3; ++k)
        if (s[k] == nullptr && cudaStreamCreateWithFlags(&s[k], cudaStreamNonBlocking) != cudaSuccess)
            return check_launch("brl_duplicate_match (capture stream)");
    *out = s;
    return BRL_OK;
}

}  // namespace brl

using namespace brl;

extern "C" {

int64_t brl_duplicate_match_scratch_bytes(int64_t n_envs, int64_t n_models) {
    if (n_envs <= 0 || n_models <= 0) return 0;
    return (int64_t)match_layout(n_envs, n_models).total;
}

long long brl_duplicate_match_graph_builds(void) {
    std::lock_guard<std::mutex> lock(cache().mu);
    return cache().builds;
}

int32_t brl_duplicate_match(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    const int64_t M = p->k_steps, P = (int64_t)p->step;
    if (M <= 0) return fail(BRL_E_OPAQUE, "brl_duplicate_match: k_steps (the pool's model count) must be > 0");
    if (b[3] == nullptr && M != 2) return fail(BRL_E_OPAQUE, "brl_duplicate_match: without env_models the pool must hold 2 nets (got %lld)", (long long)M);
    if ((b[4] != nullptr) != (P > 0))
        return fail(BRL_E_OPAQUE, "brl_duplicate_match: step (the range count, %lld) must be > 0 exactly when the range offsets are given", (long long)P);
    if (p->n_envs > INT32_MAX / 2) return fail(BRL_E_OPAQUE, "brl_duplicate_match: n_envs too large");
    if (p->n_deals <= 0) return fail(BRL_E_OPAQUE, "brl_duplicate_match: n_deals must be > 0");
    if (p->flags & BRL_F_SAMPLE) return fail(BRL_E_OPAQUE, "brl_duplicate_match: sampling is not supported (argmax only)");
    BRL_REQUIRE(b[0], "keys");
    BRL_REQUIRE(b[1], "deal_table");
    BRL_REQUIRE(b[2], "pool");
    if (b[3] != nullptr && (reinterpret_cast<uintptr_t>(b[3]) & 7u)) return fail(BRL_E_BUFFER, "brl_duplicate_match: env_models is misaligned");
    if (b[4] != nullptr && (reinterpret_cast<uintptr_t>(b[4]) & 7u)) return fail(BRL_E_BUFFER, "brl_duplicate_match: range offsets are misaligned");
    BRL_REQUIRE(b[5], "scratch");
    if (b[6] == nullptr || (reinterpret_cast<uintptr_t>(b[6]) & 3u)) return fail(BRL_E_BUFFER, "brl_duplicate_match: cum_return is NULL or misaligned");
    if (b[7] == nullptr || (reinterpret_cast<uintptr_t>(b[7]) & 7u)) return fail(BRL_E_BUFFER, "brl_duplicate_match: sums is NULL or misaligned");
    if (b[8] == nullptr || (reinterpret_cast<uintptr_t>(b[8]) & 3u)) return fail(BRL_E_BUFFER, "brl_duplicate_match: status is NULL or misaligned");
    int given = 0;
    for (int k = 9; k < 21; ++k) given += b[k] != nullptr;
    if (given != 0 && given != 12) return fail(BRL_E_BUFFER, "brl_duplicate_match: give all twelve Table_info buffers [9..20] or none");
    if (given && ((reinterpret_cast<uintptr_t>(b[10]) | reinterpret_cast<uintptr_t>(b[16])) & 15u))
        return fail(BRL_E_BUFFER, "brl_duplicate_match: Table_info rewards are not 16-byte aligned");

    MatchPlan q{};
    q.n = p->n_envs;
    q.M = (int)M;
    q.P = P;
    q.cap = brl_model_rows_capacity(q.n, M);
    q.n_deals = p->n_deals;
    q.flags = p->flags;
    q.illegal_penalty = p->illegal_penalty;
    q.illegal_bonus = p->illegal_bonus;
    q.keys = b[0];
    q.table = b[1];
    q.pool = static_cast<const unsigned char*>(b[2]);
    q.ranges = static_cast<const int64_t*>(b[4]);
    q.scratch = static_cast<unsigned char*>(b[5]);
    q.cum_return = static_cast<float*>(b[6]);
    q.sums = static_cast<double*>(b[7]);
    q.status = static_cast<int32_t*>(b[8]);
    q.L = match_layout(q.n, M);
    for (int t = 0; t < 2; ++t)
        for (int k = 0; k < 6; ++k) q.info[t][k] = given ? b[9 + 6 * t + k] : q.at(q.L.info[t][k]);
    q.default_models = b[3] == nullptr;
    q.env_models = q.default_models ? q.at<int32_t>(q.L.env_models) : static_cast<int32_t*>(b[3]);

    cudaStream_t s = (cudaStream_t)stream;
    cudaStreamCaptureStatus st;
    if (cudaStreamIsCapturing(s, &st) != cudaSuccess) return check_launch("brl_duplicate_match (capture status)");
    MatchCache& c = cache();
    std::lock_guard<std::mutex> lock(c.mu);
    cudaStream_t* side = nullptr;
    if ((rc = warm_policy_grouped_dev(!(p->flags & BRL_F_MLP_BF16))) || (rc = capture_streams(&side))) return rc;
    if (st == cudaStreamCaptureStatusActive) {  // the caller's capture: the nodes go there
        if ((rc = emit_match(q, s, side[1], side[2]))) return rc;
        return check_launch("brl_duplicate_match");
    }
    if (st != cudaStreamCaptureStatusNone) return fail(BRL_E_LAUNCH, "brl_duplicate_match: the stream's capture was invalidated");
    int dev = 0;
    cudaGetDevice(&dev);
    std::string key(reinterpret_cast<const char*>(&dev), sizeof(dev));
    key.append(reinterpret_cast<const char*>(p), sizeof(*p));
    key.append(reinterpret_cast<const char*>(b), 21 * sizeof(void*));
    auto it = c.exec.find(key);
    if (it == c.exec.end()) {
        if (cudaStreamBeginCapture(side[0], cudaStreamCaptureModeRelaxed) != cudaSuccess) return launch_error("brl_duplicate_match (capture)");
        rc = emit_match(q, side[0], side[1], side[2]);
        cudaGraph_t g = nullptr;
        const cudaError_t end = cudaStreamEndCapture(side[0], &g);
        cudaGraphExec_t exec = nullptr;
        if (rc == BRL_OK && (end != cudaSuccess || cudaGraphInstantiate(&exec, g, 0) != cudaSuccess))
            rc = launch_error("brl_duplicate_match (instantiate)");
        if (g != nullptr) cudaGraphDestroy(g);
        if (rc != BRL_OK) return rc;
        if (c.exec.size() >= kMaxCachedGraphs) {  // evict the least recently used (a graph still running is freed when it ends)
            auto lru = c.exec.begin();
            for (auto e = c.exec.begin(); e != c.exec.end(); ++e)
                if (e->second.second < lru->second.second) lru = e;
            cudaGraphExecDestroy(lru->second.first);
            c.exec.erase(lru);
        }
        it = c.exec.emplace(key, std::make_pair(exec, (uint64_t)0)).first;
        ++c.builds;
    }
    it->second.second = ++c.clock;
    if (cudaGraphLaunch(it->second.first, s) != cudaSuccess) return check_launch("brl_duplicate_match (launch)");
    return check_launch("brl_duplicate_match");
}

}  // extern "C"
