// brl_match.cu -- a whole evaluation as one stream-ordered call, its `lax.while_loop` run on the device by a CUDA graph WHILE
// node.  sm_100a only.
//   brl_duplicate_match   make_simple_duplicate_evaluate (src/evaluation.py:69-204) for every env of the batch
//   brl_evaluate_match    make_evaluate's duplicate / single-table evaluate (:207-1032) and make_simple_evaluate (:11-66):
//                         the same loop with the step log (brl_eval_act_log) and the statistics (brl_eval_summary), or with
//                         one env step per iteration and the actor's return
//   brl_call_values       brl_duplicate_match's loop with, after each forward, every live env branched on every legal call and
//                         the branches played out by a nested WHILE node (DESIGN.md f16); optionally each decision's
//                         observation and gains as training examples (DESIGN.md f17)
//
//   match start: init (brl_init) -> Table_info A / B (brl_state_fields)
//   grouping (brl_model_rows) -> control
//   WHILE (control said so) {
//       [path kernel -> IF fused forward / IF per-layer forward]    the grouped forward, sized from the device count
//       [brl_system_stats] -> brl_duplicate_step -> cum_return += rewards[:, 0] -> grouping -> control
//   }
//   match sums (brl_match_stats_ranges, or brl_match_stats for one range)
//
// All three ops share the match start and the loop (emit_while: grouping, control and a WHILE node whose body ends in
// grouping and control).  brl_evaluate_match's body adds brl_eval_act_log after the forward (full statistics), steps with
// brl_step instead of brl_duplicate_step where there is one table, and the op ends with brl_eval_summary (or nothing:
// simple).  brl_call_values' body runs a second such loop, over the branch batch, between the forward and the step.
//
// The control kernel reads the padded row count brl_model_rows left in offsets[M] and sets the loop's condition: the loop
// ends when no env is live, when a live env's net id is outside [0, M), at the loop's bound (BRL_MATCH_MAX_STEPS forwards
// for a match), or once a loop of the graph has failed; the first two failures write a status.  Nothing is read back to the
// host.  The forward path follows the host's rule (fused from kPairMinM rows on, per-layer below, unless
// BRL_F_TUNE_MLP_LAYERS / BRL_F_TUNE_MLP_FUSED pin it), applied to the device count by a path kernel and two IF nodes.
//
// On a plain stream the graph is captured on a private stream, instantiated once per set of buffers and parameters
// (cached), and launched.  On a stream that is being captured (torch.cuda.graph, an XLA command buffer) the same nodes
// go into the caller's capture.
#include <cstring>
#include <map>
#include <mutex>
#include <string>

#include "common.h"
#include "env_device.cuh"

namespace brl {

int32_t launch_policy_grouped(cudaStream_t s, int32_t flags, int64_t capacity, int n_models, const void* obs,
                              const unsigned char* pool, unsigned char* scratch, const uint8_t* mask, int32_t* action,
                              const int32_t* rows, const int32_t* block_model, const int32_t* n_rows, float* logits);
int32_t warm_policy_grouped(bool split);

// ---- kernels -----------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pair_models(int32_t* __restrict__ env_models, int64_t n) {  // every env: net 0 vs net 1
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) reinterpret_cast<int2*>(env_models)[i] = make_int2(0, 1);
}

// BRL_F_EVAL_PARTNER: every env's nets by player id (duplicate / single table: actor, partner, opponent, opponent)
__global__ void __launch_bounds__(256) k_player_models(int32_t* __restrict__ env_models, int4 ids, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) reinterpret_cast<int4*>(env_models)[i] = ids;
}

__global__ void __launch_bounds__(256) k_add_reward(float* __restrict__ cum_return, const float4* __restrict__ rewards, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) cum_return[i] += rewards[i].x;  // cum_return += state.rewards[:, 0] (src/evaluation.py:167-169)
}

// make_simple_evaluate: the actor (net 0) decides for the team of the env's initial player, the opponent (net 1) for the other
// (src/utils.py:133-202: actor, opp, actor, opp from the player to act at the quad step's start), and R gathers that player's reward
__global__ void __launch_bounds__(256) k_actor_models(int32_t* __restrict__ env_models, int8_t* __restrict__ actor,
                                                      const int8_t* __restrict__ player, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int8_t p = player[i];
    actor[i] = p;
    reinterpret_cast<int2*>(env_models)[i] = p < 2 ? make_int2(0, 1) : make_int2(1, 0);
}

// k_actor_models with a partner, by player id: the initial player p plays net 0, its partner p ^ 1 net 2, the other team net 1
__global__ void __launch_bounds__(256) k_actor_partner_models(int32_t* __restrict__ env_models, int8_t* __restrict__ actor,
                                                              const int8_t* __restrict__ player, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int8_t p = player[i];
    actor[i] = p;
    const int own = p & 1 ? 2 : 0, other = 2 - own;  // player ids 0/1 and 2/3 are partners
    reinterpret_cast<int4*>(env_models)[i] = p < 2 ? make_int4(own, other, 1, 1) : make_int4(1, 1, own, other);
}

__global__ void __launch_bounds__(256) k_add_actor_reward(float* __restrict__ R, const float* __restrict__ rewards,
                                                          const int8_t* __restrict__ actor, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) R[i] += rewards[4 * i + actor[i]];  // R + rewards[actor] (src/evaluation.py:60); non-zero on the last step only
}

__global__ void __launch_bounds__(256) k_sum_rewards(float* __restrict__ cum_return, float4* __restrict__ rewards_sum,
                                                     const float4* __restrict__ rewards, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 r = rewards[i];
    float4 s = rewards_sum[i];
    s.x += r.x;
    s.y += r.y;
    s.z += r.z;
    s.w += r.w;
    rewards_sum[i] = s;  // rewards += state.rewards, cum_return += rewards[:, 0] (src/evaluation.py:407-411)
    cum_return[i] += r.x;
}

// after each grouping: continue while rows are live; stop with a status on a bad net id or at the step bound, and stop once a
// loop of the graph has failed (brl_call_values' two loops share the status; a BRL_MATCH_RECORD_CAPACITY status does not stop
// them: the sums stay complete).  `iter` counts the forwards the loop has been allowed to run.
__global__ void k_match_control(const int32_t* __restrict__ n_rows, int32_t* __restrict__ iter, int32_t* __restrict__ status,
                                cudaGraphConditionalHandle loop, int bound) {
    const int rows = *n_rows, it = *iter, st = *status;
    bool go = rows > 0 && st != BRL_MATCH_BAD_MODEL && st != BRL_MATCH_STEP_BOUND;
    if (rows < 0) {
        *status = BRL_MATCH_BAD_MODEL;
    } else if (go && it >= bound) {
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

// ---- brl_call_values (env_device.cuh, DESIGN.md f16) ----------------------------------------------------------------------
// one thread per branch slot j = 38 i + a of base env i: the slot's state is S_i, to be stepped with call a by brl_step; a
// slot whose env is finished or whose call is illegal is born finished (a no-op step, never listed by brl_model_rows).  The
// slot's nets by player id come from the env's (by team: expanded); r[j] = 0; the slot loop's iteration counter restarts.
template <int kStride>
__global__ void __launch_bounds__(256) k_branch_calls(const uint4* __restrict__ state, const uint8_t* __restrict__ done,
                                                      const int32_t* __restrict__ env_models, uint4* __restrict__ br_state,
                                                      int32_t* __restrict__ br_action, int4* __restrict__ br_models,
                                                      float* __restrict__ r, int32_t* __restrict__ br_iter, int64_t n) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nb = n * kNumActions;
    if (j == 0) *br_iter = 0;
    if (j >= nb) return;
    const int64_t i = j / kNumActions;
    const int a = (int)(j - i * kNumActions);
    Env e;
    load_env(state, n, i, e);
    if (done[i] != 0 || !((env_legal_mask(e) >> a) & 1ull)) e.A |= kTermBit;
    store_env(br_state, nb, j, e);
    br_action[j] = a;
    r[j] = 0.0f;
    const int32_t* m = env_models + kStride * i;
    br_models[j] = kStride == 4 ? make_int4(m[0], m[1], m[2], m[3]) : make_int4(m[0], m[0], m[1], m[1]);
}

// One thread per live base env after its branches ended: the decision's gains and regret into the int64 sums of its net,
// context and played call (integer atomics: exact and order-independent), the invariant r(played) = R_T, and a record.
struct CvOut {
    unsigned long long *gain, *regret, *mismatch, *count;  // gain_sums[M,75,38,38,4], regret_sums[M,75,4], mismatch[M], count[1]
    int32_t *env, *table, *player, *net, *context, *played;  // records (NULL: none)
    float* r;                                                // records' r[cap, 38]
    int64_t cap, env_offset;
    int32_t* status;
};

template <int kStride>
__global__ void __launch_bounds__(256) k_call_value_gains(const uint4* __restrict__ state, const uint8_t* __restrict__ done,
                                                          const int32_t* __restrict__ env_models, const int32_t* __restrict__ action,
                                                          const uint8_t* __restrict__ a_done, const float4* __restrict__ ra,
                                                          const float4* __restrict__ rb, const float* __restrict__ r, CvOut o,
                                                          int64_t n, int n_models) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || done[i] != 0) return;
    Env e;
    load_env(state, n, i, e);
    const uint32_t p = f_player_at(e, f_cur_seat(e));
    const int m = env_models[kStride * i + (kStride == 4 ? (int)p : (p < 2u ? 0 : 1))];
    const int b = action[i];
    if (m < 0 || m >= n_models || b < 0 || b >= kNumActions) return;
    const uint32_t c = system_context(system_prefix(e));
    const uint64_t legal = env_legal_mask(e);
    const int t = a_done[i] != 0;  // table A has ended: this is table B
    const float R_a = ra[i].x, R_b = rb[i].x, R_other = t ? R_a : R_b;
    const float base = imp_of_difference(R_a + R_b);
    const float* ri = r + i * kNumActions;
    unsigned long long* gm = o.gain + (((size_t)m * kSysContexts + c) * kNumActions + b) * kNumActions * kCvStats;
    int32_t regret = INT32_MIN;
    for (int a = 0; a < kNumActions; ++a) {
        if (!((legal >> a) & 1ull)) continue;
        const long long g = call_value_gain(ri[a], R_other, base, p < 2u);
        regret = max(regret, (int32_t)g);
        unsigned long long* cell = gm + a * kCvStats;
        atomicAdd(cell, 1ull);
        atomicAdd(cell + 1, (unsigned long long)g);
        atomicAdd(cell + 2, (unsigned long long)(g * g));
        if (g > 0) atomicAdd(cell + 3, 1ull);
    }
    unsigned long long* rg = o.regret + ((size_t)m * kSysContexts + c) * kCvStats;
    atomicAdd(rg, 1ull);
    atomicAdd(rg + 1, (unsigned long long)(long long)regret);
    atomicAdd(rg + 2, (unsigned long long)((long long)regret * regret));
    if (regret > 0) atomicAdd(rg + 3, 1ull);
    if (ri[b] != (t ? R_b : R_a)) atomicAdd(o.mismatch + m, 1ull);
    if (o.env == nullptr) return;
    const unsigned long long k = atomicAdd(o.count, 1ull);
    if ((long long)k >= o.cap) {
        atomicCAS(o.status, BRL_MATCH_OK, BRL_MATCH_RECORD_CAPACITY);
        return;
    }
    o.env[k] = (int32_t)(o.env_offset + i);
    o.table[k] = t;
    o.player[k] = (int32_t)p;
    o.net[k] = m;
    o.context[k] = (int32_t)c;
    o.played[k] = b;
    for (int a = 0; a < kNumActions; ++a) o.r[k * kNumActions + a] = (legal >> a) & 1ull ? ri[a] : __int_as_float(0x7fc00000);
}

// Training examples of the records (DESIGN.md f17), in the graph only with buffers [19] / [20].  k_cv_mark saves the record
// count before an iteration's k_call_value_gains; k_cv_examples then fills the slots that kernel took, [saved, min(count,
// cap)), one warp per slot: the base env's bf16 observation row (what the forward of this iteration read: the branches
// step their own buffers) and the gains of the record's r, NaN where r is (an illegal call).
__global__ void k_cv_mark(const unsigned long long* __restrict__ count, unsigned long long* __restrict__ saved) { *saved = *count; }

__global__ void __launch_bounds__(256) k_cv_examples(const uint4* __restrict__ obs, const float4* __restrict__ ra,
                                                     const float4* __restrict__ rb, const CvOut o,
                                                     const unsigned long long* __restrict__ saved, uint4* __restrict__ ex_obs,
                                                     float* __restrict__ ex_gain) {
    constexpr int kRow = BRL_OBS_DIM * 2 / 16;  // one bf16 row in 16-byte words
    const int lane = threadIdx.x & 31;
    const unsigned long long end = min(*o.count, (unsigned long long)o.cap);
    const unsigned long long k = *saved + (((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (k >= end) return;
    const int64_t i = (int64_t)o.env[k] - o.env_offset;
    for (int w = lane; w < kRow; w += 32) ex_obs[k * kRow + w] = obs[i * kRow + w];
    const float R_a = ra[i].x, R_b = rb[i].x, R_other = o.table[k] ? R_a : R_b;
    const float base = imp_of_difference(R_a + R_b);
    const bool team1 = o.player[k] < 2;
    for (int a = lane; a < kNumActions; a += 32) {
        const float r = o.r[k * kNumActions + a];
        ex_gain[k * kNumActions + a] = isnan(r) ? r : (float)call_value_gain(r, R_other, base, team1);
    }
}

// ---- the scratch ----------------------------------------------------------------------------------------------------------
// brl_duplicate_match's pieces; brl_evaluate_match (mode > 0) appends its own behind them
struct MatchLayout {
    size_t state, obs, mask, rewards, terminated, player, action, info[2][6], env_models, rows, counts, offsets, block_model, ctl,
        forward, logits, fields[6], rewards_sum, actor, total;
};

static MatchLayout match_layout(int64_t n, int64_t M, int mode = 0, bool player_models = false) {
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
    L.env_models = take(un * (player_models ? 16 : 8));
    L.rows = take(cap * 4);
    L.counts = take((size_t)M * 4);
    L.offsets = take((size_t)(M + 1) * 4);
    L.block_model = take(cap / kGroupRows * 4);
    L.ctl = take(16);  // i32 iteration counter
    L.forward = take((size_t)brl_policy_grouped_scratch_bytes(n, M));
    if (mode == BRL_EVAL_MATCH_DUPLICATE || mode == BRL_EVAL_MATCH_SINGLE) {
        L.logits = take(un * BRL_NUM_ACTIONS * 4);
        for (int k = 0; k < 4; ++k) L.fields[k] = take(un * 4);  // i32 step_count, last_bid, last_bidder, pass_num
        for (int k = 4; k < 6; ++k) L.fields[k] = take(un);      // u8 call_x, call_xx
    }
    if (mode == BRL_EVAL_MATCH_SINGLE) L.rewards_sum = take(un * 16);
    if (mode == BRL_EVAL_MATCH_SIMPLE) L.actor = take(un);
    L.total = off;
    return L;
}

// every device pointer and size one match needs
struct MatchPlan {
    const char* who;  // the op, for error messages
    int mode;         // 0: brl_duplicate_match; else BRL_EVAL_MATCH_*
    bool free_run;    // brl_evaluate_match: team 2 always passes
    bool partner;     // brl_evaluate_match: BRL_F_EVAL_PARTNER
    bool player_models;  // env_models[n, 4] by player id (BRL_F_PLAYER_MODELS)
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
    void *state, *obs, *mask, *terminated, *player;  // the loop's env buffers: the scratch's, or the caller's final-state outputs
    float* logits;       // full statistics: the acting net's logits by env, for brl_eval_act_log (else NULL)
    float* acc;          // full statistics: the per-env log rows
    float* rewards_sum;  // single table: sum of the step rewards
    uint32_t* system_hist;  // brl_duplicate_match [21]: bidding-system histogram of each decision (NULL: not counted)
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

// check_launch for one step of `who`
static int32_t launched(const char* who, const char* step) {
    const cudaError_t err = cudaGetLastError();
    return err == cudaSuccess ? BRL_OK : fail(BRL_E_LAUNCH, "%s (%s): %s", who, step, cudaGetErrorString(err));
}

// a failed graph-building call: its CUDA error, or a plain failure when the call left none
static int32_t launch_error(const char* who, const char* step) {
    const int32_t rc = launched(who, step);
    return rc != BRL_OK ? rc : fail(BRL_E_LAUNCH, "%s (%s) failed", who, step);
}

static unsigned blocks(int64_t n) { return (unsigned)((n + 255) / 256); }

static int32_t model_rows(const MatchPlan& q, cudaStream_t s) {
    void* b[7] = {q.player, q.terminated, q.env_models, q.at(q.L.rows), q.at(q.L.counts), q.offsets(), q.at(q.L.block_model)};
    BrlParams p = env_params(q, q.n);
    p.k_steps = q.M;
    if (q.player_models) p.flags |= BRL_F_PLAYER_MODELS;
    return brl_model_rows(s, b, &p, sizeof(p));
}

static int32_t control(const MatchPlan& q, cudaStream_t s, cudaGraphConditionalHandle loop, int bound) {
    k_match_control<<<1, 1, 0, s>>>(q.offsets() + q.M, q.at<int32_t>(q.L.ctl), q.status, loop, bound);
    return launched(q.who, "control");
}

// the capture's graph, with the stream's current dependencies; a conditional node of `type` there (its body in *body), made
// the stream's only dependency
static int32_t add_conditional(const char* who, cudaStream_t s, cudaGraphConditionalHandle h, cudaGraphConditionalNodeType type,
                               cudaGraph_t* body) {
    cudaStreamCaptureStatus st;
    cudaGraph_t g = nullptr;
    const cudaGraphNode_t* deps = nullptr;
    size_t n_deps = 0;
    if (cudaStreamGetCaptureInfo(s, &st, nullptr, &g, &deps, &n_deps) != cudaSuccess || st != cudaStreamCaptureStatusActive)
        return launch_error(who, "capture info");
    cudaGraphNodeParams cp{};
    cp.type = cudaGraphNodeTypeConditional;
    cp.conditional.handle = h;
    cp.conditional.type = type;
    cp.conditional.size = 1;
    cudaGraphNode_t node;
    if (cudaGraphAddNode(&node, g, deps, n_deps, &cp) != cudaSuccess ||
        cudaStreamUpdateCaptureDependencies(s, &node, 1, cudaStreamSetCaptureDependencies) != cudaSuccess)
        return launch_error(who, "conditional node");
    *body = cp.conditional.phGraph_out[0];
    return BRL_OK;
}

static int32_t new_handle(const char* who, cudaStream_t s, cudaGraphConditionalHandle* h) {
    cudaStreamCaptureStatus st;
    cudaGraph_t g = nullptr;
    if (cudaStreamGetCaptureInfo(s, &st, nullptr, &g) != cudaSuccess || st != cudaStreamCaptureStatusActive ||
        cudaGraphConditionalHandleCreate(h, g, 0, cudaGraphCondAssignDefault) != cudaSuccess)
        return launch_error(who, "conditional handle");
    return BRL_OK;
}

// fill `body` by capturing what `fn(side)` enqueues on the side stream
template <class F>
static int32_t capture_into(const char* who, cudaGraph_t body, cudaStream_t side, F&& fn) {
    if (cudaStreamBeginCaptureToGraph(side, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed) != cudaSuccess)
        return launch_error(who, "body capture");
    const int32_t rc = fn(side);
    cudaGraph_t out = nullptr;
    const cudaError_t end = cudaStreamEndCapture(side, &out);
    if (rc != BRL_OK) return rc;
    if (end != cudaSuccess) return launch_error(who, "body capture");
    return BRL_OK;
}

// a loop over q's envs on s: grouping and control, then a WHILE node whose body (captured on s_body) is what `body` enqueues
// followed by grouping and control.  The loop runs at most `bound` times.
template <class F>
static int32_t emit_while(const MatchPlan& q, cudaStream_t s, cudaStream_t s_body, int bound, F&& body) {
    int32_t rc;
    cudaGraphConditionalHandle loop;
    cudaGraph_t g;
    if ((rc = new_handle(q.who, s, &loop)) || (rc = model_rows(q, s)) || (rc = control(q, s, loop, bound)) ||
        (rc = add_conditional(q.who, s, loop, cudaGraphCondTypeWhile, &g)))
        return rc;
    return capture_into(q.who, g, s_body, [&](cudaStream_t sb) {
        int32_t r;
        if ((r = body(sb)) || (r = model_rows(q, sb))) return r;
        return control(q, sb, loop, bound);
    });
}

static int32_t forward(const MatchPlan& q, cudaStream_t s, int32_t path_flag) {
    const int32_t flags = (q.flags & BRL_F_MLP_BF16) | path_flag;
    return launch_policy_grouped(s, flags, q.cap, q.M, q.obs, q.pool, q.at<unsigned char>(q.L.forward), static_cast<uint8_t*>(q.mask),
                                 q.at<int32_t>(q.L.action), q.at<int32_t>(q.L.rows), q.at<int32_t>(q.L.block_model),
                                 q.offsets() + q.M, q.logits);
}

// brl_step without auto-reset on one table (:406; make_simple_evaluate: src/utils.py:133-202 one sub-step at a time)
static int32_t table_step(const MatchPlan& q, cudaStream_t s) {
    const BrlParams p = env_params(q, q.n);
    void* b[10] = {q.state, q.at(q.L.action), const_cast<void*>(q.table), q.state, q.obs, q.mask, q.at(q.L.rewards), q.terminated,
                   q.player, nullptr};
    return brl_step(s, b, &p, sizeof(p));
}

// the env step of one iteration: brl_duplicate_step on both tables (:164, :772-774), or one table's step
static int32_t env_step(const MatchPlan& q, cudaStream_t s) {
    if (q.mode == BRL_EVAL_MATCH_SINGLE || q.mode == BRL_EVAL_MATCH_SIMPLE) return table_step(q, s);
    const BrlParams p = env_params(q, q.n);
    void* b[21] = {q.state, q.at(q.L.action), const_cast<void*>(q.table)};
    for (int t = 0; t < 2; ++t)
        for (int k = 0; k < 6; ++k) b[3 + 6 * t + k] = q.info[t][k];
    b[15] = q.state;
    b[16] = q.obs;
    b[17] = q.mask;
    b[18] = q.at(q.L.rewards);
    b[19] = q.terminated;
    b[20] = q.player;
    return brl_duplicate_step(s, b, &p, sizeof(p));
}

// one iteration of the loop (src/evaluation.py:124-169; :388-411 / :748-777 with the step log; :42-61), on the body's capture
// stream s1; s2 captures the IF bodies
// the grouped forward of one iteration on s1: the pinned path, or the path kernel and an IF node per path (bodies captured on s2)
static int32_t emit_forward(const MatchPlan& q, cudaStream_t s1, cudaStream_t s2) {
    if (q.flags & BRL_F_TUNE_MLP_LAYERS) return forward(q, s1, BRL_F_TUNE_MLP_LAYERS);
    if (q.flags & BRL_F_TUNE_MLP_FUSED) return forward(q, s1, BRL_F_TUNE_MLP_FUSED);
    int32_t rc;
    cudaGraphConditionalHandle h_fused, h_layers;
    if ((rc = new_handle(q.who, s1, &h_fused)) || (rc = new_handle(q.who, s1, &h_layers))) return rc;
    k_match_path<<<1, 1, 0, s1>>>(q.offsets() + q.M, h_fused, h_layers);
    if ((rc = launched(q.who, "path"))) return rc;
    cudaGraph_t body;
    if ((rc = add_conditional(q.who, s1, h_fused, cudaGraphCondTypeIf, &body)) ||
        (rc = capture_into(q.who, body, s2, [&](cudaStream_t s) { return forward(q, s, BRL_F_TUNE_MLP_FUSED); })) ||
        (rc = add_conditional(q.who, s1, h_layers, cudaGraphCondTypeIf, &body)) ||
        (rc = capture_into(q.who, body, s2, [&](cudaStream_t s) { return forward(q, s, BRL_F_TUNE_MLP_LAYERS); })))
        return rc;
    return BRL_OK;
}

static int32_t emit_body(const MatchPlan& q, cudaStream_t s1, cudaStream_t s2) {
    int32_t rc = emit_forward(q, s1, s2);
    if (rc != BRL_OK) return rc;
    if (q.acc) {  // the acting team's masked argmax and update_log_info; free-run: team 2 passes, its forwarded rows unread
        void* b[7] = {q.logits, q.free_run ? nullptr : q.logits, q.mask, q.player, q.terminated, q.at(q.L.action), q.acc};
        BrlParams p{};
        p.n_envs = q.n;
        p.flags = q.mode == BRL_EVAL_MATCH_SINGLE ? BRL_F_EVAL_INDICATOR_BIDS : 0;
        if ((rc = brl_eval_act_log(s1, b, &p, sizeof(p)))) return rc;
    }
    if (q.system_hist) {  // each live env's decision, in the state before the step
        void* b[6] = {q.state, const_cast<void*>(q.table), q.at(q.L.action), q.terminated, q.env_models, q.system_hist};
        BrlParams p = env_params(q, q.n);
        p.k_steps = q.M;
        p.flags = q.player_models ? BRL_F_PLAYER_MODELS : 0;
        if ((rc = brl_system_stats(s1, b, &p, sizeof(p)))) return rc;
    }
    if ((rc = env_step(q, s1))) return rc;
    if (q.mode == BRL_EVAL_MATCH_SIMPLE)
        k_add_actor_reward<<<blocks(q.n), 256, 0, s1>>>(q.cum_return, q.at<float>(q.L.rewards), q.at<int8_t>(q.L.actor), q.n);
    else if (q.mode == BRL_EVAL_MATCH_SINGLE)
        k_sum_rewards<<<blocks(q.n), 256, 0, s1>>>(q.cum_return, reinterpret_cast<float4*>(q.rewards_sum), q.at<float4>(q.L.rewards), q.n);
    else
        k_add_reward<<<blocks(q.n), 256, 0, s1>>>(q.cum_return, q.at<float4>(q.L.rewards), q.n);
    return launched(q.who, "cum_return");
}

// brl_evaluate_match's end: the final state's fields and every log_info sum (src/evaluation.py:448-596, :839-1027)
static int32_t emit_summary(const MatchPlan& q, cudaStream_t s) {
    void* f[6];
    for (int k = 0; k < 6; ++k) f[k] = q.at(q.L.fields[k]);
    const bool single = q.mode == BRL_EVAL_MATCH_SINGLE;
    void* bf[12] = {q.state, nullptr, nullptr, nullptr, nullptr, single ? f[1] : nullptr, single ? f[2] : nullptr,
                    single ? f[4] : nullptr, single ? f[5] : nullptr, single ? f[3] : nullptr, f[0], nullptr};
    BrlParams p = env_params(q, q.n);
    int32_t rc;
    if ((rc = brl_state_fields(s, bf, &p, sizeof(p)))) return rc;
    void* bs[16] = {q.acc, q.cum_return, f[0]};
    if (single) {  // table A = the final state's fields (no rewards: the sign comes from cum_return), no table B
        bs[3] = f[1];
        bs[4] = f[2];
        bs[5] = f[4];
        bs[6] = f[5];
        bs[8] = f[3];
    } else {       // both Table_infos: last_bid, last_bidder, call_x, call_xx, rewards
        for (int t = 0; t < 2; ++t) {
            bs[3 + 6 * t] = q.info[t][2];
            bs[4 + 6 * t] = q.info[t][3];
            bs[5 + 6 * t] = q.info[t][4];
            bs[6 + 6 * t] = q.info[t][5];
            bs[7 + 6 * t] = q.info[t][1];
        }
    }
    bs[15] = q.sums;
    BrlParams ps{};
    ps.n_envs = q.n;
    return brl_eval_summary(s, bs, &ps, sizeof(ps));
}

// the envs from the keys (src/evaluation.py:93-95, observation in bf16: what the forward reads) and, where the plan has
// Table_infos, Table_info A = B = the init state's terminated, rewards, last_bid, last_bidder, call_x, call_xx (:97-112)
static int32_t match_start(const MatchPlan& q, cudaStream_t s) {
    void* bi[8] = {const_cast<void*>(q.keys), const_cast<void*>(q.table), q.state, q.obs, q.mask, q.at(q.L.rewards), q.terminated,
                   q.player};
    const BrlParams p = env_params(q, q.n);
    int32_t rc;
    if ((rc = brl_init(s, bi, &p, sizeof(p)))) return rc;
    if (q.mode != 0 && q.mode != BRL_EVAL_MATCH_DUPLICATE) return BRL_OK;
    void* bf[12] = {q.state, nullptr, nullptr, nullptr, nullptr, q.info[0][2], q.info[0][3], q.info[0][4], q.info[0][5]};
    if ((rc = brl_state_fields(s, bf, &p, sizeof(p)))) return rc;
    const size_t un = (size_t)q.n, bytes[6] = {un, un * 16, un * 4, un * 4, un, un};
    if (cudaMemcpyAsync(q.info[0][0], q.terminated, bytes[0], cudaMemcpyDeviceToDevice, s) != cudaSuccess ||
        cudaMemcpyAsync(q.info[0][1], q.at(q.L.rewards), bytes[1], cudaMemcpyDeviceToDevice, s) != cudaSuccess)
        return launched(q.who, "Table_info");
    for (int k = 0; k < 6; ++k)
        if (cudaMemcpyAsync(q.info[1][k], q.info[0][k], bytes[k], cudaMemcpyDeviceToDevice, s) != cudaSuccess)
            return launched(q.who, "Table_info");
    return BRL_OK;
}

// the whole match on the capturing stream s0 (its own capture, or the caller's)
static int32_t emit_match(const MatchPlan& q, cudaStream_t s0, cudaStream_t s1, cudaStream_t s2) {
    int32_t rc;
    const size_t un = (size_t)q.n;
    if (cudaMemsetAsync(q.status, 0, sizeof(int32_t), s0) != cudaSuccess ||
        cudaMemsetAsync(q.at(q.L.ctl), 0, sizeof(int32_t), s0) != cudaSuccess ||
        cudaMemsetAsync(q.cum_return, 0, un * sizeof(float), s0) != cudaSuccess ||
        cudaMemsetAsync(q.at(q.L.action), 0, un * sizeof(int32_t), s0) != cudaSuccess ||  // finished envs keep a (no-op) Pass
        (q.acc && cudaMemsetAsync(q.acc, 0, un * BRL_EVAL_ACC_COLS * sizeof(float), s0) != cudaSuccess) ||
        (q.logits && cudaMemsetAsync(q.logits, 0, un * BRL_NUM_ACTIONS * sizeof(float), s0) != cudaSuccess) ||
        (q.rewards_sum && cudaMemsetAsync(q.rewards_sum, 0, un * 16, s0) != cudaSuccess) ||
        (q.free_run && !q.partner && cudaMemsetAsync(q.env_models, 0, un * 8, s0) != cudaSuccess))  // free-run: net 0 forwards every row
        return launched(q.who, "memset");
    if (q.partner && q.mode != BRL_EVAL_MATCH_SIMPLE)  // free-run: net 0 forwards team 2's rows, team 1's split between nets 0 / 2
        k_player_models<<<blocks(q.n), 256, 0, s0>>>(q.env_models, q.free_run ? make_int4(0, 2, 0, 0) : make_int4(0, 2, 1, 1), q.n);
    else if (q.default_models)
        k_pair_models<<<blocks(q.n), 256, 0, s0>>>(q.env_models, q.n);
    if ((rc = match_start(q, s0))) return rc;
    if (q.mode == BRL_EVAL_MATCH_SIMPLE) {
        if (q.partner)
            k_actor_partner_models<<<blocks(q.n), 256, 0, s0>>>(q.env_models, q.at<int8_t>(q.L.actor), static_cast<const int8_t*>(q.player),
                                                                q.n);
        else
            k_actor_models<<<blocks(q.n), 256, 0, s0>>>(q.env_models, q.at<int8_t>(q.L.actor), static_cast<const int8_t*>(q.player), q.n);
        if ((rc = launched(q.who, "actor"))) return rc;
    }
    if ((rc = emit_while(q, s0, s1, BRL_MATCH_MAX_STEPS, [&](cudaStream_t s) { return emit_body(q, s, s2); }))) return rc;
    if (q.mode == BRL_EVAL_MATCH_SIMPLE) return BRL_OK;  // the output is R itself
    if (q.mode != 0) return emit_summary(q, s0);
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
    cudaStream_t streams[kMaxDevices][4] = {};
    uint64_t clock = 0;
    long long builds = 0;
};
static MatchCache& cache() {
    static MatchCache* c = new MatchCache();  // never destroyed: instantiated graphs outlive static destruction order
    return *c;
}
constexpr size_t kMaxCachedGraphs = 16;

static int32_t capture_streams(const char* who, cudaStream_t** out) {
    cudaStream_t* s = cache().streams[device_slot()];
    for (int k = 0; k < 4; ++k)
        if (s[k] == nullptr && cudaStreamCreateWithFlags(&s[k], cudaStreamNonBlocking) != cudaSuccess)
            return launched(who, "capture stream");
    *out = s;
    return BRL_OK;
}

// run what `emit(s0, s1, s2)` enqueues on `stream`: into the caller's capture when the stream is being captured, else by
// (building and caching, keyed by the op, its params and its n_buffers buffer addresses, then) launching its graph
template <class Emit>
static int32_t run_graph(const char* who, cudaStream_t s, const BrlParams* p, void** b, int n_buffers, Emit&& emit) {
    int32_t rc;
    cudaStreamCaptureStatus st;
    if (cudaStreamIsCapturing(s, &st) != cudaSuccess) return launched(who, "capture status");
    MatchCache& c = cache();
    std::lock_guard<std::mutex> lock(c.mu);
    cudaStream_t* side = nullptr;
    if ((rc = warm_policy_grouped(!(p->flags & BRL_F_MLP_BF16))) || (rc = capture_streams(who, &side))) return rc;
    if (st == cudaStreamCaptureStatusActive) {  // the caller's capture: the nodes go there
        if ((rc = emit(s, side))) return rc;
        return check_launch(who);
    }
    if (st != cudaStreamCaptureStatusNone) return fail(BRL_E_LAUNCH, "%s: the stream's capture was invalidated", who);
    int dev = 0;
    cudaGetDevice(&dev);
    std::string key(who);
    key.append(reinterpret_cast<const char*>(&dev), sizeof(dev));
    key.append(reinterpret_cast<const char*>(p), sizeof(*p));
    key.append(reinterpret_cast<const char*>(b), n_buffers * sizeof(void*));
    auto it = c.exec.find(key);
    if (it == c.exec.end()) {
        if (cudaStreamBeginCapture(side[0], cudaStreamCaptureModeRelaxed) != cudaSuccess) return launch_error(who, "capture");
        rc = emit(side[0], side);
        cudaGraph_t g = nullptr;
        const cudaError_t end = cudaStreamEndCapture(side[0], &g);
        cudaGraphExec_t exec = nullptr;
        if (rc == BRL_OK && (end != cudaSuccess || cudaGraphInstantiate(&exec, g, 0) != cudaSuccess))
            rc = launch_error(who, "instantiate");
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
    if (cudaGraphLaunch(it->second.first, s) != cudaSuccess) return launched(who, "launch");
    return check_launch(who);
}

static int32_t run_match(const MatchPlan& q, cudaStream_t s, const BrlParams* p, void** b, int n_buffers) {
    return run_graph(q.who, s, p, b, n_buffers, [&](cudaStream_t s0, cudaStream_t* side) {
        return emit_match(q, s0, side[1], side[2]);
    });
}

// the plan's fields every mode shares; the env buffers and Table_infos start in the scratch
static MatchPlan base_plan(const char* who, int mode, const BrlParams* p, int64_t M, void* scratch, bool player_models = false) {
    MatchPlan q{};
    q.who = who;
    q.mode = mode;
    q.n = p->n_envs;
    q.M = (int)M;
    q.cap = brl_model_rows_capacity(q.n, M);
    q.n_deals = p->n_deals;
    q.flags = p->flags;
    q.illegal_penalty = p->illegal_penalty;
    q.illegal_bonus = p->illegal_bonus;
    q.scratch = static_cast<unsigned char*>(scratch);
    q.player_models = player_models;
    q.L = match_layout(q.n, M, mode, player_models);
    for (int t = 0; t < 2; ++t)
        for (int k = 0; k < 6; ++k) q.info[t][k] = q.at(q.L.info[t][k]);
    q.state = q.at(q.L.state);
    q.obs = q.at(q.L.obs);
    q.mask = q.at(q.L.mask);
    q.terminated = q.at(q.L.terminated);
    q.player = q.at(q.L.player);
    q.env_models = q.at<int32_t>(q.L.env_models);
    return q;
}

// how many of b[from, to) are given: an all-or-none group has none or to - from
static int given(void* const* b, int from, int to) {
    int k = 0;
    for (int i = from; i < to; ++i) k += b[i] != nullptr;
    return k;
}

// the names of a Table_info A / B pair of buffers, in buffer order
#define BRL_TABLE_INFO_NAMES                                                                                                  \
    "table_a.terminated", "table_a.rewards", "table_a.last_bid", "table_a.last_bidder", "table_a.call_x", "table_a.call_xx",  \
        "table_b.terminated", "table_b.rewards", "table_b.last_bid", "table_b.last_bidder", "table_b.call_x", "table_b.call_xx"

// ---- brl_call_values ----------------------------------------------------------------------------------------------------
constexpr int kAuctionMaxCalls = BRL_MATCH_MAX_STEPS / 2;  // the bound of one branch's auction

// the scratch: the base match's pieces, then a branch batch of 38 n slots (brl_duplicate_match's pieces for 38 n envs with
// nets by player id), then the slots' r
static size_t cv_branch_at(int64_t n, int64_t M) { return match_layout(n, M).total; }
static size_t cv_r_at(int64_t n, int64_t M) { return cv_branch_at(n, M) + match_layout(n * kNumActions, M, 0, true).total; }
static size_t cv_scratch_bytes(int64_t n, int64_t M) { return cv_r_at(n, M) + (size_t)n * kNumActions * 4; }

struct CvPlan {
    MatchPlan q, br;  // the base match (its Table_infos in the scratch) and the branch batch
    const float4 *ra, *rb;
    float* r;
    CvOut o;
    uint4* ex_obs;    // [19] training examples' bf16 obs[cap, 480] (NULL: none)
    float* ex_gain;   // [20] their f32 gain[cap, 38]
    unsigned long long* saved;  // the record count before the iteration's gains: a spare word of the base loop's ctl
};

// one step of the branch batch, then r += rewards[:, 0] (non-zero on a slot's last step only)
static int32_t branch_step(const CvPlan& c, cudaStream_t s) {
    const MatchPlan& br = c.br;
    int32_t rc;
    if ((rc = table_step(br, s))) return rc;
    k_add_reward<<<blocks(br.n), 256, 0, s>>>(c.r, br.at<float4>(br.L.rewards), br.n);
    return launched(br.who, "branch reward");
}

// one base iteration: forward -> branch every live env on every legal call -> play the branches out (nested WHILE) -> gains
// -> brl_duplicate_step
static int32_t emit_cv_body(const CvPlan& c, cudaStream_t s1, cudaStream_t s2, cudaStream_t s3) {
    const MatchPlan &q = c.q, &br = c.br;
    int32_t rc;
    if ((rc = emit_forward(q, s1, s2))) return rc;
    const uint4* state = static_cast<const uint4*>(q.state);
    const uint8_t* done = static_cast<const uint8_t*>(q.terminated);
    if (q.player_models)
        k_branch_calls<4><<<blocks(br.n), 256, 0, s1>>>(state, done, q.env_models, static_cast<uint4*>(br.state), br.at<int32_t>(br.L.action),
                                                       reinterpret_cast<int4*>(br.env_models), c.r, br.at<int32_t>(br.L.ctl), q.n);
    else
        k_branch_calls<2><<<blocks(br.n), 256, 0, s1>>>(state, done, q.env_models, static_cast<uint4*>(br.state), br.at<int32_t>(br.L.action),
                                                       reinterpret_cast<int4*>(br.env_models), c.r, br.at<int32_t>(br.L.ctl), q.n);
    // the branches' auctions to their ends: the forward's IF nodes sit one level deeper here, in the nested WHILE's body
    if ((rc = launched(q.who, "branch calls")) || (rc = branch_step(c, s1)) ||
        (rc = emit_while(br, s1, s2, kAuctionMaxCalls, [&](cudaStream_t s) {
             int32_t r2;
             if ((r2 = emit_forward(br, s, s3))) return r2;
             return branch_step(c, s);
         })))
        return rc;
    const int32_t* action = q.at<int32_t>(q.L.action);
    const uint8_t* a_done = static_cast<const uint8_t*>(q.info[0][0]);
    if (c.ex_obs) k_cv_mark<<<1, 1, 0, s1>>>(c.o.count, c.saved);
    if (q.player_models)
        k_call_value_gains<4><<<blocks(q.n), 256, 0, s1>>>(state, done, q.env_models, action, a_done, c.ra, c.rb, c.r, c.o, q.n, q.M);
    else
        k_call_value_gains<2><<<blocks(q.n), 256, 0, s1>>>(state, done, q.env_models, action, a_done, c.ra, c.rb, c.r, c.o, q.n, q.M);
    if (c.ex_obs)  // at most one record per base env and iteration: n warps
        k_cv_examples<<<blocks(q.n * 32), 256, 0, s1>>>(static_cast<const uint4*>(q.obs), c.ra, c.rb, c.o, c.saved, c.ex_obs,
                                                         c.ex_gain);
    if ((rc = launched(q.who, "gains"))) return rc;
    return env_step(q, s1);
}

// the whole op on s0: zeroed outputs, the match start of brl_duplicate_match, then the base loop
static int32_t emit_call_values(const CvPlan& c, cudaStream_t s0, cudaStream_t s1, cudaStream_t s2, cudaStream_t s3) {
    const MatchPlan& q = c.q;
    const size_t un = (size_t)q.n, cells = (size_t)q.M * kSysContexts * kNumActions * kNumActions * kCvStats * 8;
    int32_t rc;
    if (cudaMemsetAsync(q.status, 0, sizeof(int32_t), s0) != cudaSuccess ||
        cudaMemsetAsync(q.at(q.L.ctl), 0, sizeof(int32_t), s0) != cudaSuccess ||
        cudaMemsetAsync(q.at(q.L.action), 0, un * sizeof(int32_t), s0) != cudaSuccess ||
        cudaMemsetAsync(c.o.gain, 0, cells, s0) != cudaSuccess ||
        cudaMemsetAsync(c.o.regret, 0, (size_t)q.M * kSysContexts * kCvStats * 8, s0) != cudaSuccess ||
        cudaMemsetAsync(c.o.mismatch, 0, (size_t)q.M * 8, s0) != cudaSuccess ||
        (c.o.count && cudaMemsetAsync(c.o.count, 0, 8, s0) != cudaSuccess))
        return launched(q.who, "memset");
    if ((rc = match_start(q, s0))) return rc;
    return emit_while(q, s0, s1, BRL_MATCH_MAX_STEPS, [&](cudaStream_t s) { return emit_cv_body(c, s, s2, s3); });
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
    const bool player_models = (p->flags & BRL_F_PLAYER_MODELS) != 0;
    if (M <= 0) return fail(BRL_E_OPAQUE, "brl_duplicate_match: k_steps (the pool's model count) must be > 0");
    if (player_models && b[3] == nullptr)
        return fail(BRL_E_BUFFER, "brl_duplicate_match: BRL_F_PLAYER_MODELS needs env_models [3] (i32[n, 4])");
    if (b[3] == nullptr && M != 2) return fail(BRL_E_OPAQUE, "brl_duplicate_match: without env_models the pool must hold 2 nets (got %lld)", (long long)M);
    if ((b[4] != nullptr) != (P > 0))
        return fail(BRL_E_OPAQUE, "brl_duplicate_match: step (the range count, %lld) must be > 0 exactly when the range offsets are given", (long long)P);
    if (p->n_envs > INT32_MAX / 2) return fail(BRL_E_OPAQUE, "brl_duplicate_match: n_envs too large");
    if (p->n_deals <= 0) return fail(BRL_E_OPAQUE, "brl_duplicate_match: n_deals must be > 0");
    if (p->flags & BRL_F_SAMPLE) return fail(BRL_E_OPAQUE, "brl_duplicate_match: sampling is not supported (argmax only)");
    static const char* names[22] = {"keys", "deal_table", "pool", "env_models", "range offsets", "scratch", "cum_return", "sums",
                                    "status", BRL_TABLE_INFO_NAMES, "system histogram [21]"};
    static const uint8_t align[22] = {16, 16, 16, 8, 8, 16, 4, 8, 4, 0, 16, 0, 0, 0, 0, 0, 16, 0, 0, 0, 0, 4};
    const unsigned nullable = 1u << 3 | 1u << 4 | 0xFFFu << 9 | 1u << 21;
    // problems are reported in buffer order: the Table_info group [9..20] before the optional histogram [21]
    if ((rc = check_buffers("brl_duplicate_match", b, names, 21, nullable, 0u, align))) return rc;
    const int tables = given(b, 9, 21);
    if (tables != 0 && tables != 12) return fail(BRL_E_BUFFER, "brl_duplicate_match: give all twelve Table_info buffers [9..20] or none");
    if ((rc = check_buffers("brl_duplicate_match", b, names, 22, nullable, 0u, align))) return rc;

    MatchPlan q = base_plan("brl_duplicate_match", 0, p, M, b[5]);
    q.P = P;
    q.keys = b[0];
    q.table = b[1];
    q.pool = static_cast<const unsigned char*>(b[2]);
    q.ranges = static_cast<const int64_t*>(b[4]);
    q.cum_return = static_cast<float*>(b[6]);
    q.sums = static_cast<double*>(b[7]);
    q.status = static_cast<int32_t*>(b[8]);
    if (tables)
        for (int t = 0; t < 2; ++t)
            for (int k = 0; k < 6; ++k) q.info[t][k] = b[9 + 6 * t + k];
    q.default_models = b[3] == nullptr;
    q.player_models = player_models;  // the caller's env_models; the scratch keeps its [n, 2] layout
    if (!q.default_models) q.env_models = static_cast<int32_t*>(b[3]);
    q.system_hist = static_cast<uint32_t*>(b[21]);
    return run_match(q, (cudaStream_t)stream, p, b, 22);
}

int64_t brl_evaluate_match_scratch_bytes(int64_t n_envs, int64_t mode) {
    if (n_envs <= 0 || mode < BRL_EVAL_MATCH_DUPLICATE || mode > BRL_EVAL_MATCH_SIMPLE) return 0;
    return (int64_t)match_layout(n_envs, 2, (int)mode).total;
}

int64_t brl_evaluate_match_partner_scratch_bytes(int64_t n_envs, int64_t mode) {
    if (n_envs <= 0 || mode < BRL_EVAL_MATCH_DUPLICATE || mode > BRL_EVAL_MATCH_SIMPLE) return 0;
    return (int64_t)match_layout(n_envs, 3, (int)mode, true).total;
}

int32_t brl_evaluate_match(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    const int mode = BRL_EVAL_MATCH_MODE(p->flags);
    const bool free_run = (p->flags & BRL_F_EVAL_FREE_RUN) != 0, full = mode != BRL_EVAL_MATCH_SIMPLE;
    if (mode < BRL_EVAL_MATCH_DUPLICATE || mode > BRL_EVAL_MATCH_SIMPLE)
        return fail(BRL_E_OPAQUE, "brl_evaluate_match: flags name no mode (BRL_F_EVAL_MATCH(BRL_EVAL_MATCH_*))");
    if (free_run && !full) return fail(BRL_E_OPAQUE, "brl_evaluate_match: BRL_F_EVAL_FREE_RUN is a mode of the full-statistics evaluation");
    const bool partner = (p->flags & BRL_F_EVAL_PARTNER) != 0;
    if (partner && p->k_steps != 3)
        return fail(BRL_E_OPAQUE, "brl_evaluate_match: BRL_F_EVAL_PARTNER needs a pool of 3 nets, k_steps = 3 (got %lld)", (long long)p->k_steps);
    if (p->n_envs > INT32_MAX / 2) return fail(BRL_E_OPAQUE, "brl_evaluate_match: n_envs too large");
    if (p->n_deals <= 0) return fail(BRL_E_OPAQUE, "brl_evaluate_match: n_deals must be > 0");
    if (p->flags & BRL_F_SAMPLE) return fail(BRL_E_OPAQUE, "brl_evaluate_match: sampling is not supported (argmax only)");
    // buffers a mode does not read are not checked: acc and sums in simple mode, the Table_infos outside duplicate mode and the
    // final state outside single-table mode
    static const char* names[26] = {"keys", "deal_table", "pool", "scratch", "cum_return", "acc", "sums", "status", BRL_TABLE_INFO_NAMES,
                                    "final state", "observation", "mask", "rewards", "terminated", "current_player"};
    const bool dup = mode == BRL_EVAL_MATCH_DUPLICATE, single = mode == BRL_EVAL_MATCH_SINGLE;
    const uint8_t t16 = dup ? 16 : 0, f16 = single ? 16 : 0;
    const uint8_t align[26] = {16, 16, 16, 16, 4, full ? 4 : 0, full ? 8 : 0, 4, 0, t16, 0, 0, 0, 0, 0, t16, 0, 0, 0, 0,
                               f16, f16, single ? 2 : 0, f16, 0, 0};
    const unsigned nullable = (full ? 0u : 1u << 5 | 1u << 6) | 0xFFFu << 8 | 0x3Fu << 20;
    if ((rc = check_buffers("brl_evaluate_match", b, names, 26, nullable, 0u, align))) return rc;
    const int tables = dup ? given(b, 8, 20) : 0, finals = single ? given(b, 20, 26) : 0;
    if (tables != 0 && tables != 12) return fail(BRL_E_BUFFER, "brl_evaluate_match: give all twelve Table_info buffers [8..19] or none");
    if (finals != 0 && finals != 6) return fail(BRL_E_BUFFER, "brl_evaluate_match: give all six final-state buffers [20..25] or none");

    MatchPlan q = base_plan("brl_evaluate_match", mode, p, partner ? 3 : 2, b[3], partner);
    q.free_run = free_run;
    q.partner = partner;
    q.keys = b[0];
    q.table = b[1];
    q.pool = static_cast<const unsigned char*>(b[2]);
    q.cum_return = static_cast<float*>(b[4]);
    q.status = static_cast<int32_t*>(b[7]);
    q.default_models = mode != BRL_EVAL_MATCH_SIMPLE && !free_run;
    if (full) {
        q.acc = static_cast<float*>(b[5]);
        q.sums = static_cast<double*>(b[6]);
        q.logits = q.at<float>(q.L.logits);
    }
    if (tables)
        for (int t = 0; t < 2; ++t)
            for (int k = 0; k < 6; ++k) q.info[t][k] = b[8 + 6 * t + k];
    if (single) {
        q.rewards_sum = q.at<float>(q.L.rewards_sum);
        if (finals) {
            q.state = b[20];
            q.obs = b[21];
            q.mask = b[22];
            q.rewards_sum = static_cast<float*>(b[23]);
            q.terminated = b[24];
            q.player = b[25];
        }
    }
    return run_match(q, (cudaStream_t)stream, p, b, 26);
}

}  // extern "C"

extern "C" {

int64_t brl_call_values_scratch_bytes(int64_t n_envs, int64_t n_models) {
    if (n_envs <= 0 || n_models <= 0) return 0;
    return (int64_t)cv_scratch_bytes(n_envs, n_models);
}

int32_t brl_call_values(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    const int64_t M = p->k_steps, cap = (int64_t)p->seed;
    const bool player_models = (p->flags & BRL_F_PLAYER_MODELS) != 0;
    if (M <= 0) return fail(BRL_E_OPAQUE, "brl_call_values: k_steps (the pool's model count) must be > 0");
    if (p->n_envs > INT32_MAX / 2 / kNumActions) return fail(BRL_E_OPAQUE, "brl_call_values: n_envs too large");
    if (p->n_deals <= 0) return fail(BRL_E_OPAQUE, "brl_call_values: n_deals must be > 0");
    if (p->flags & BRL_F_SAMPLE) return fail(BRL_E_OPAQUE, "brl_call_values: sampling is not supported (argmax only)");
    if (cap < 0) return fail(BRL_E_OPAQUE, "brl_call_values: the record capacity (seed) must be >= 0");
    static const char* names[21] = {"keys", "deal_table", "pool", "env_models", "rewards_a", "rewards_b", "scratch", "gain_sums",
                                    "regret_sums", "mismatch", "status", "count", "env", "table", "player", "net", "context", "played",
                                    "r", "obs", "gain"};
    static const uint8_t align[21] = {16, 0, 16, 16, 16, 16, 16, 8, 8, 8, 4, 8, 4, 4, 4, 4, 4, 4, 4, 16, 4};
    // problems are reported in buffer order: the record group [11..18] before the optional examples [19], [20]
    if ((rc = check_buffers("brl_call_values", b, names, 19, 0x3FFu << 11, 0u, align))) return rc;
    const int records = given(b, 11, 19);
    if (records != 0 && records != 8) return fail(BRL_E_BUFFER, "brl_call_values: give all eight record buffers [11..18] or none");
    if ((rc = check_buffers("brl_call_values", b, names, 21, 0x3FFu << 11, 0u, align))) return rc;
    const bool examples = b[19] != nullptr;
    if (examples != (b[20] != nullptr))
        return fail(BRL_E_BUFFER, "brl_call_values: give both training-example buffers [19] obs and [20] gain, or neither");
    if (examples && !records) return fail(BRL_E_BUFFER, "brl_call_values: the training examples [19], [20] need the eight record buffers [11..18]");

    CvPlan c{};
    c.q = base_plan("brl_call_values", 0, p, M, b[6]);
    c.q.keys = b[0];
    c.q.table = b[1];
    c.q.pool = static_cast<const unsigned char*>(b[2]);
    c.q.player_models = player_models;
    c.q.env_models = static_cast<int32_t*>(b[3]);
    c.q.status = static_cast<int32_t*>(b[10]);
    BrlParams pb = *p;
    pb.n_envs = p->n_envs * kNumActions;
    c.br = base_plan("brl_call_values", 0, &pb, M, static_cast<unsigned char*>(b[6]) + cv_branch_at(p->n_envs, M), true);
    c.br.table = b[1];
    c.br.pool = c.q.pool;
    c.br.status = c.q.status;
    c.ra = static_cast<const float4*>(b[4]);
    c.rb = static_cast<const float4*>(b[5]);
    c.r = reinterpret_cast<float*>(static_cast<unsigned char*>(b[6]) + cv_r_at(p->n_envs, M));
    c.o.gain = static_cast<unsigned long long*>(b[7]);
    c.o.regret = static_cast<unsigned long long*>(b[8]);
    c.o.mismatch = static_cast<unsigned long long*>(b[9]);
    c.o.status = c.q.status;
    c.o.cap = cap;
    c.o.env_offset = p->env_offset;
    if (records) {
        c.o.count = static_cast<unsigned long long*>(b[11]);
        c.o.env = static_cast<int32_t*>(b[12]);
        c.o.table = static_cast<int32_t*>(b[13]);
        c.o.player = static_cast<int32_t*>(b[14]);
        c.o.net = static_cast<int32_t*>(b[15]);
        c.o.context = static_cast<int32_t*>(b[16]);
        c.o.played = static_cast<int32_t*>(b[17]);
        c.o.r = static_cast<float*>(b[18]);
    }
    if (examples) {
        c.ex_obs = static_cast<uint4*>(b[19]);
        c.ex_gain = static_cast<float*>(b[20]);
        c.saved = reinterpret_cast<unsigned long long*>(c.q.at<unsigned char>(c.q.L.ctl) + 8);  // ctl holds one i32 in 16 bytes
    }
    // the cache key holds all 21 addresses: a graph with the example kernels and one without are two entries
    return run_graph(c.q.who, (cudaStream_t)stream, p, b, 21, [&](cudaStream_t s0, cudaStream_t* side) {
        return emit_call_values(c, s0, side[1], side[2], side[3]);
    });
}

}  // extern "C"
