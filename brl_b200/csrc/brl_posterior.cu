// brl_posterior.cu -- hand reading (DESIGN.md f18, restated by tests/posterior_ref.py): the hidden hands an auction implies
// under the nets' own policies, by self-normalised importance sampling of the 39 cards the observer cannot see, and by
// resample-move sequential Monte Carlo over the calls of the prefix (brl_hand_posterior_smc, DESIGN.md f19, tests/smc_ref.py).
//
//   brl_hand_posterior   check pass -> segment counts -> row layout -> row list / block nets -> public pass -> sampler ->
//                        observation expansion -> grouped forward (launch_policy_grouped, logits out) -> log-likelihood ->
//                        per-query reduction
//
// A segment (j, k) is call k of query j made by a seat other than the observer: N consecutive rows, one per sample, in the
// group of the net of the caller.  Net m's segments are ordered by (j, k); its group starts at group_off[m] and is padded to
// kGroupRows rows, so every row block of the forward runs one net.  Every count the layout needs is computed on the device,
// and the padded row count is left in device memory for the forward; nothing is read back.
#include <cuda_bf16.h>

#include "common.h"
#include "env_device.cuh"
#include "obs_row.cuh"

namespace brl {

int32_t launch_policy_grouped(cudaStream_t s, int32_t flags, int64_t capacity, int n_models, const void* obs,
                              const unsigned char* pool, unsigned char* scratch, const uint8_t* mask, int32_t* action,
                              const int32_t* rows, const int32_t* block_model, const int32_t* n_rows, float* logits);
int32_t warm_policy_grouped(bool split);

constexpr uint32_t kPostSeating = 0u | (1u << 2) | (2u << 4) | (3u << 6);  // player ids = seats
constexpr int kPostCards = 3 * 52;                                           // cards[j, 3, 52]
constexpr int kPostOutputs = kPostCards + 3 * BRL_POST_FEATURES;             // + features[j, 3, 95]
constexpr int kPostChunk = 256;                                              // samples staged per step of the reduction

// the public part of one segment: the caller's observation without its hand, its legal mask and its call
struct PostSeg {
    uint32_t R[14];  // observation words 0..13 rotated to the caller, vulnerability bits set, hand bits clear
    uint32_t legal_lo, legal_hi;
    int32_t call, query, seat, pad;
};

struct PostArgs {
    const uint8_t* table;
    const uint8_t* calls;
    const int64_t* offsets;
    const int32_t* board;
    const int8_t* dealer;
    const uint8_t* vul;
    const int32_t* query;      // [Q, 3] = (t, s, L)
    const int32_t* seat_nets;  // [Q, 4]
    int32_t* status;           // [Q]
    int32_t* meta;             // [0] padded row count  [1] the layout exceeds the capacity
    int64_t* group_off;        // [M + 1] first row of net m's group
    int64_t* seg_prefix;       // [M + 1] first segment index of net m
    int32_t* totals;           // [M] segments of net m
    int32_t* base;             // [Q, 4] segments of the caller's net in the queries before j
    PostSeg* seg;
    int32_t* rows;
    int32_t* block_model;
    void* obs;                 // bf16 [capacity, 480]
    const float* logits;       // [capacity, 38]
    uint64_t* hands;           // [Q, N, 4]
    double* logw;              // [Q, N]
    double* cards;
    double* features;
    double* weights;
    int64_t Q, cap, g0;
    uint64_t seed;
    int32_t N, M, n_deals;
    float tau;
};

struct PostQuery {
    int64_t off;
    int32_t len, s, L, row, dealer, vul;
};

__device__ __forceinline__ PostQuery post_query(const PostArgs& a, int64_t j) {
    PostQuery q;
    const int32_t t = a.query[3 * j];
    q.s = a.query[3 * j + 1];
    q.L = a.query[3 * j + 2];
    q.off = a.offsets[t];
    q.len = (int32_t)(a.offsets[t + 1] - q.off);
    q.row = a.board ? a.board[t] : t;
    q.dealer = a.dealer ? (int32_t)(a.dealer[t] & 3) : 0;
    q.vul = a.vul ? (int32_t)(a.vul[t] & 3) : 0;
    return q;
}

// calls of seat `seat` among calls 0 .. L-1 (call k by seat (dealer + k) mod 4)
__device__ __forceinline__ int32_t calls_by(int32_t seat, int32_t dealer, int32_t L) {
    const int32_t r = (seat - dealer) & 3;
    return L > r ? (L - 1 - r) / 4 + 1 : 0;
}

__device__ __forceinline__ void post_reset(Env& e, const PostQuery& q) {
    env_reset(e, (uint32_t)q.row, (uint32_t)q.dealer, (uint32_t)q.vul & 1u, (uint32_t)q.vul >> 1, kPostSeating, 0ull);
}

struct NoHand {  // env_observe_words without the observer's hand (the sampled hand is OR'd in per row)
    __device__ __forceinline__ uint64_t hand(uint32_t, uint32_t) const { return 0ull; }
};

// ---- 1. check pass: one block per query, one thread per call of the prefix ------------------------------------------------
__global__ void __launch_bounds__(128) k_post_check(const PostArgs a) {
    __shared__ int first;
    const int64_t j = blockIdx.x;
    const PostQuery q = post_query(a, j);
    if (threadIdx.x == 0) {
        int code = BRL_POST_OK;
        if (q.s < 0 || q.s > 3 || q.L < 0 || q.row < 0 || q.row >= a.n_deals) code = BRL_POST_BAD_QUERY;
        else if (q.L > q.len) code = BRL_POST_SHORT;
        else
            for (int sg = 0; sg < 4; ++sg) {
                const int32_t m = a.seat_nets[4 * j + sg];
                if (sg != q.s && calls_by(sg, q.dealer, q.L) > 0 && (m < 0 || m >= a.M)) code = BRL_POST_BAD_NET;
            }
        first = code == BRL_POST_OK ? 0x7FFFFFFF : code;  // a query-level failure comes first
    }
    __syncthreads();
    if (first == 0x7FFFFFFF)
        for (int32_t k = threadIdx.x; k < q.L; k += blockDim.x) {
            Env e;
            post_reset(e, q);
            for (int32_t c = 0; c < k; ++c) env_step(e, (int32_t)a.calls[q.off + c], TableRows{a.table}, -1.0f, 1.0f);
            const int32_t c = (int32_t)a.calls[q.off + k];
            int code = BRL_POST_OK;
            if (f_terminated(e)) code = BRL_POST_SHORT;
            else if (c < 0 || c >= kNumActions || !((env_legal_mask(e) >> c) & 1ull)) code = BRL_POST_ILLEGAL;
            if (code != BRL_POST_OK) atomicMin(&first, 8 + 8 * k + code);  // the earliest failing call
        }
    __syncthreads();
    if (threadIdx.x == 0) a.status[j] = first == 0x7FFFFFFF ? BRL_POST_OK : (first < 8 ? first : (first & 7));
}

// Which calls of a query are in a forward: calls(j, s, sg, dealer, L) counts seat sg's calls in the row set (sg != s), and
// takes(j, s, k, sg) says whether call k (by sg != s) is one of them.  f18 reads every call of the prefix; brl_hand_posterior_smc
// reads one stage's call, or a move's two seats up to its stage (SmcWindow below).
struct AllCalls {
    __device__ __forceinline__ int32_t calls(int64_t, int32_t, int32_t sg, int32_t dealer, int32_t L) const {
        return calls_by(sg, dealer, L);
    }
    __device__ __forceinline__ bool takes(int64_t, int32_t, int32_t, int32_t) const { return true; }
};

// the kernels take their row set as an optional trailing parameter: none is AllCalls (f18's parameter block is unchanged)
__device__ __forceinline__ AllCalls row_set() { return AllCalls{}; }
template <class Rows>
__device__ __forceinline__ Rows row_set(const Rows& r) { return r; }

// ---- 2. segment counts: block m scans the queries for net m's segments ----------------------------------------------------
__device__ __forceinline__ int32_t block_exclusive_scan(int32_t v, int32_t* warp_tot, int32_t* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[warp] = x;
    __syncthreads();
    if (warp == 0) {
        int32_t w = lane < nw ? warp_tot[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int32_t y = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += y;
        }
        if (lane < nw) warp_tot[lane] = w;  // inclusive
        if (lane == nw - 1) *total = w;
    }
    __syncthreads();
    const int32_t r = (warp ? warp_tot[warp - 1] : 0) + x - v;
    __syncthreads();
    return r;
}

template <class... Sel>
__global__ void __launch_bounds__(1024) k_post_count(const PostArgs a, const Sel... sel) {
    const auto rows = row_set(sel...);
    __shared__ int32_t warp_tot[32];
    __shared__ int32_t total;
    const int32_t m = blockIdx.x;
    int32_t carry = 0;
    for (int64_t c0 = 0; c0 < a.Q; c0 += blockDim.x) {
        const int64_t j = c0 + threadIdx.x;
        int32_t cnt = 0, s = -1, L = 0, dealer = 0;
        int4 nets = make_int4(-1, -1, -1, -1);
        if (j < a.Q && a.status[j] == BRL_POST_OK) {
            s = a.query[3 * j + 1];
            L = a.query[3 * j + 2];
            const int32_t t = a.query[3 * j];
            dealer = a.dealer ? (int32_t)(a.dealer[t] & 3) : 0;
            nets = reinterpret_cast<const int4*>(a.seat_nets)[j];
            const int32_t n4[4] = {nets.x, nets.y, nets.z, nets.w};
            for (int sg = 0; sg < 4; ++sg)
                if (sg != s && n4[sg] == m) cnt += rows.calls(j, s, sg, dealer, L);
        }
        const int32_t ex = block_exclusive_scan(cnt, warp_tot, &total);
        if (s >= 0) {
            const int32_t n4[4] = {nets.x, nets.y, nets.z, nets.w};
            for (int sg = 0; sg < 4; ++sg)
                if (sg != s && n4[sg] == m) a.base[4 * j + sg] = carry + ex;
        }
        carry += total;
    }
    if (threadIdx.x == 0) a.totals[m] = carry;
}

// ---- 3. layout: group offsets, the padded row count, the capacity check ---------------------------------------------------
__global__ void k_post_layout(const PostArgs a) {
    int64_t off = 0, segs = 0;
    for (int m = 0; m < a.M; ++m) {
        a.group_off[m] = off;
        a.seg_prefix[m] = segs;
        const int64_t rows = (int64_t)a.totals[m] * a.N;
        off += (rows + kGroupRows - 1) / kGroupRows * kGroupRows;
        segs += a.totals[m];
    }
    a.group_off[a.M] = off;
    a.seg_prefix[a.M] = segs;
    const bool over = off > a.cap;
    a.meta[0] = over ? 0 : (int32_t)off;
    a.meta[1] = over ? 1 : 0;
}

// ---- 4. the forward's row list (identity, -1 on a group's padding) and each row block's net -------------------------------
__device__ __forceinline__ int post_group(const PostArgs& a, int64_t r) {
    int m = 0;
    while (m + 1 < a.M && a.group_off[m + 1] <= r) ++m;
    return m;
}

__global__ void __launch_bounds__(256) k_post_rows(const PostArgs a) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.meta[0]) return;
    const int m = post_group(a, r);
    a.rows[r] = r - a.group_off[m] < (int64_t)a.totals[m] * a.N ? (int32_t)r : -1;
    if ((r & (kGroupRows - 1)) == 0) a.block_model[r / kGroupRows] = m;
}

// ---- 5. public pass: one block per query, one thread per call of the prefix -----------------------------------------------
template <class... Sel>
__global__ void __launch_bounds__(128) k_post_public(const PostArgs a, const Sel... sel) {
    const auto rows = row_set(sel...);
    const int64_t j = blockIdx.x;
    if (a.status[j] != BRL_POST_OK || a.meta[1]) return;
    const PostQuery q = post_query(a, j);
    const int4 nv = reinterpret_cast<const int4*>(a.seat_nets)[j];
    const int32_t nets[4] = {nv.x, nv.y, nv.z, nv.w};
    for (int32_t k = threadIdx.x; k < q.L; k += blockDim.x) {
        const int32_t sg = (q.dealer + k) & 3;
        if (sg == q.s || !rows.takes(j, q.s, k, sg)) continue;
        const int32_t m = nets[sg];
        int32_t rank = 0;  // earlier segments of this query in net m's group
        for (int32_t c = 0; c < k; ++c) {
            const int32_t sc = (q.dealer + c) & 3;
            rank += sc != q.s && nets[sc] == m && rows.takes(j, q.s, c, sc);
        }
        Env e;
        post_reset(e, q);
        for (int32_t c = 0; c < k; ++c) env_step(e, (int32_t)a.calls[q.off + c], TableRows{a.table}, -1.0f, 1.0f);
        uint32_t R[kObsWords];
        env_observe_words(e, NoHand{}, (uint32_t)sg, R);
        const uint64_t legal = env_legal_mask(e);
        PostSeg& d = a.seg[a.seg_prefix[m] + a.base[4 * j + sg] + rank];
#pragma unroll
        for (int w = 0; w < 14; ++w) d.R[w] = R[w];
        d.legal_lo = (uint32_t)legal;
        d.legal_hi = (uint32_t)(legal >> 32);
        d.call = (int32_t)a.calls[q.off + k];
        d.query = (int32_t)j;
        d.seat = sg;
        d.pad = 0;
    }
}

// ---- 6. sampler: one thread per (query, sample) ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_post_sample(const PostArgs a) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.Q * a.N) return;
    const int64_t j = idx / a.N;
    const uint32_t i = (uint32_t)(idx - j * a.N);
    ulonglong2* out = reinterpret_cast<ulonglong2*>(a.hands + 4 * idx);
    if (a.status[j] == BRL_POST_BAD_QUERY) {
        out[0] = make_ulonglong2(0ull, 0ull);
        out[1] = make_ulonglong2(0ull, 0ull);
        return;
    }
    const PostQuery q = post_query(a, j);
    const uint64_t own = TableRows{a.table}.hand((uint32_t)q.row, (uint32_t)q.s);
    uint8_t h[39];
    int n = 0;
    for (int c = 0; c < 52; ++c)
        if (!((own >> c) & 1ull) && n < 39) h[n++] = (uint8_t)c;
    const uint64_t g = (uint64_t)(a.g0 + j);
    const uint2 key = make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32));
    uint4 u = make_uint4(0u, 0u, 0u, 0u);
    for (int t = 0; t < 38; ++t) {
        if ((t & 3) == 0) u = philox4x32(make_uint4((uint32_t)g, (uint32_t)(g >> 32), BRL_POST_TAG + (uint32_t)(t >> 2), i), key);
        const uint32_t w = (t & 3) == 0 ? u.x : ((t & 3) == 1 ? u.y : ((t & 3) == 2 ? u.z : u.w));
        const int hi = 38 - t;
        const int lo = (int)__umulhi(w, (uint32_t)(hi + 1));
        const uint8_t x = h[hi];
        h[hi] = h[lo];
        h[lo] = x;
    }
    uint64_t hand[4];
    hand[q.s] = own;
    for (int r = 0; r < 3; ++r) {
        uint64_t m = 0ull;
        for (int c = 0; c < 13; ++c) m |= 1ull << h[13 * r + c];
        hand[(q.s + 1 + r) & 3] = m;
    }
    out[0] = make_ulonglong2(hand[0], hand[1]);
    out[1] = make_ulonglong2(hand[2], hand[3]);
}

// ---- 7. observation expansion: one warp per row -----------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_post_expand(const PostArgs a) {
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= a.meta[0]) return;
    const int m = a.block_model[r / kGroupRows];
    const int64_t local = r - a.group_off[m];
    if (local >= (int64_t)a.totals[m] * a.N) return;  // padding: the forward gathers zeros for row -1
    const PostSeg& d = a.seg[a.seg_prefix[m] + local / a.N];
    const int64_t i = local % a.N;
    const uint64_t hand = a.hands[((int64_t)d.query * a.N + i) * 4 + d.seat];
    uint32_t R[kObsWords];
#pragma unroll
    for (int w = 0; w < 14; ++w) R[w] = d.R[w];
    R[13] |= (uint32_t)(hand << 12);  // observation bits 428..447
    R[14] = (uint32_t)(hand >> 20);   // observation bits 448..479
    emit_obs_row<kObsBF16>(R, threadIdx.x & 31, a.obs, r);
}

// ---- 8. log-likelihood: one thread per (query, sample), the query's segments in k order ------------------------------------
// k_post_loglik's two terms as functions, for the SMC kernels (k_post_loglik keeps them inline: its code is unchanged)
// the masked first argmax of a logits row, kNumActions when nothing is legal
__device__ __forceinline__ int post_argmax(const float* l, uint64_t legal) {
    float best = -INFINITY;
    int arg = kNumActions;
    for (int x = 0; x < kNumActions; ++x)
        if (((legal >> x) & 1ull) && l[x] > best) { best = l[x]; arg = x; }
    return arg;
}

// the f32 log-softmax over the legal calls of l / tau at call c (tau > 0)
__device__ __forceinline__ float post_log_softmax(const float* l, uint64_t legal, int32_t c, float tau) {
    float mx = -INFINITY;
    for (int x = 0; x < kNumActions; ++x)
        if ((legal >> x) & 1ull) mx = fmaxf(mx, l[x] / tau);
    float se = 0.0f;
    for (int x = 0; x < kNumActions; ++x)
        if ((legal >> x) & 1ull) se += expf(l[x] / tau - mx);
    return l[c] / tau - mx - logf(se);
}

__global__ void __launch_bounds__(256) k_post_loglik(const PostArgs a) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.Q * a.N) return;
    const int64_t j = idx / a.N, i = idx - j * a.N;
    if (a.status[j] != BRL_POST_OK || a.meta[1]) {
        a.logw[idx] = __longlong_as_double(0x7FF8000000000000ll);
        return;
    }
    const int32_t t = a.query[3 * j], s = a.query[3 * j + 1], L = a.query[3 * j + 2];
    const int32_t dealer = a.dealer ? (int32_t)(a.dealer[t] & 3) : 0;
    const int4 nv = reinterpret_cast<const int4*>(a.seat_nets)[j];
    const int32_t nets[4] = {nv.x, nv.y, nv.z, nv.w};
    int32_t seen[4] = {0, 0, 0, 0};  // segments so far per net, counted at the first seat holding that net
    double sum = 0.0;
    for (int32_t k = 0; k < L && sum != -INFINITY; ++k) {
        const int32_t sg = (dealer + k) & 3;
        if (sg == s) continue;
        const int32_t m = nets[sg];
        int al = 0;
        while (nets[al] != m) ++al;
        const int64_t rank = (int64_t)a.base[4 * j + sg] + seen[al]++;
        const PostSeg& d = a.seg[a.seg_prefix[m] + rank];
        const uint64_t legal = (uint64_t)d.legal_lo | ((uint64_t)d.legal_hi << 32);
        const float* l = a.logits + (a.group_off[m] + rank * a.N + i) * kNumActions;
        const int32_t c = d.call;
        if (a.tau == 0.0f) {
            float best = -INFINITY;
            int arg = kNumActions;
            for (int x = 0; x < kNumActions; ++x)
                if (((legal >> x) & 1ull) && l[x] > best) { best = l[x]; arg = x; }
            if (arg != c) sum = -INFINITY;
        } else {
            float mx = -INFINITY;
            for (int x = 0; x < kNumActions; ++x)
                if ((legal >> x) & 1ull) mx = fmaxf(mx, l[x] / a.tau);
            float se = 0.0f;
            for (int x = 0; x < kNumActions; ++x)
                if ((legal >> x) & 1ull) se += expf(l[x] / a.tau - mx);
            sum += (double)(l[c] / a.tau - mx - logf(se));
        }
    }
    a.logw[idx] = sum;
}

// ---- 9. reduction: one block per query ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(512) k_post_reduce(const PostArgs a) {
    __shared__ double wsh[kPostChunk];
    __shared__ uint64_t hsh[3][kPostChunk];
    __shared__ uint8_t fsh[3][kPostChunk][6];  // hcp, four suit lengths, balanced
    __shared__ double red[16];
    const int64_t j = blockIdx.x;
    const int tid = threadIdx.x;
    const double nan = __longlong_as_double(0x7FF8000000000000ll);
    int st = a.status[j];
    if (a.meta[1]) st = BRL_POST_CAPACITY;
    double mx = -INFINITY;
    if (st == BRL_POST_OK)
        for (int64_t i = tid; i < a.N; i += blockDim.x) mx = fmax(mx, a.logw[j * a.N + i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((tid & 31) == 0) red[tid >> 5] = mx;
    __syncthreads();
    mx = -INFINITY;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) mx = fmax(mx, red[w]);
    double* cards = a.cards + j * kPostCards;
    double* feat = a.features + j * 3 * BRL_POST_FEATURES;
    double* wt = a.weights + 4 * j;
    if (tid == 0 && a.meta[1]) a.status[j] = BRL_POST_CAPACITY;
    if (st != BRL_POST_OK || mx == -INFINITY) {
        for (int o = tid; o < kPostOutputs; o += blockDim.x) {
            if (o < kPostCards) cards[o] = nan;
            else feat[o - kPostCards] = nan;
        }
        if (tid == 0) {
            wt[0] = wt[1] = wt[2] = nan;
            wt[3] = 0.0;
        }
        return;
    }
    const int s = a.query[3 * j + 1];
    double acc = 0.0, W = 0.0, W2 = 0.0, count = 0.0;
    for (int64_t c0 = 0; c0 < a.N; c0 += kPostChunk) {
        const int n = (int)min((int64_t)kPostChunk, a.N - c0);
        if (tid < n) {
            const int64_t i = c0 + tid;
            const double lw = a.logw[j * a.N + i];
            wsh[tid] = exp(lw - mx);
            const uint64_t* hs = a.hands + (j * a.N + i) * 4;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                const uint64_t h = hs[(s + 1 + r) & 3];
                const HandFeatures f = hand_features(h);
                hsh[r][tid] = h;
                fsh[r][tid][0] = (uint8_t)f.hcp;
#pragma unroll
                for (int u = 0; u < 4; ++u) fsh[r][tid][1 + u] = (uint8_t)f.len[u];
                fsh[r][tid][5] = (uint8_t)f.balanced;
            }
        }
        __syncthreads();
        if (tid < kPostCards) {
            const int r = tid / 52, c = tid % 52;
            for (int x = 0; x < n; ++x)
                if ((hsh[r][x] >> c) & 1ull) acc += wsh[x];
        } else if (tid < kPostOutputs) {
            const int r = (tid - kPostCards) / BRL_POST_FEATURES, col = (tid - kPostCards) % BRL_POST_FEATURES;
            const int slot = col < 38 ? 0 : (col < 94 ? 1 + (col - 38) / 14 : 5);
            const int want = col < 38 ? col : (col < 94 ? (col - 38) % 14 : 1);
            for (int x = 0; x < n; ++x)
                if (fsh[r][x][slot] == want) acc += wsh[x];
        } else if (tid == kPostOutputs) {
            for (int x = 0; x < n; ++x) {
                const double w = wsh[x];
                W += w;
                W2 += w * w;
                count += w > 0.0 ? 1.0 : 0.0;
            }
        }
        __syncthreads();
    }
    if (tid == kPostOutputs) {
        red[0] = W;
        wt[0] = mx;
        wt[1] = W;
        wt[2] = W2;
        wt[3] = count;
    }
    __syncthreads();
    W = red[0];
    if (tid < kPostCards) cards[tid] = acc / W;
    else if (tid < kPostOutputs) feat[tid - kPostCards] = acc / W;
}

// ---- brl_hand_posterior_smc: resample-move SMC over the calls of the prefix (DESIGN.md f19, restated by tests/smc_ref.py) ----
//   check -> sampler -> init -> per stage k: [reweight forward -> reweight -> ESS test / resample -> gather ->
//   R x (propose -> move forward -> accept)] -> end -> f18's reduction -> finish
// Stage k's rows are call k of every live query (SmcWindow with move < 0); move mv's rows are the calls <= k of the two seats
// of the move's pair, for the queries that resampled at stage k.  Both run through f18's layout with that row set.
constexpr uint8_t kSmcLive = 1;   // status OK and some particle with w > 0
constexpr uint8_t kSmcMoved = 2;  // resampled at the current stage: its particles move

struct SmcArgs {
    uint8_t* flags;                  // [Q] kSmc*
    double* ell;                     // [Q, N, 3] per hidden seat (LHO, partner, RHO) sums of l_k
    double* tmp_ell;
    uint64_t* tmp_hands;
    uint64_t* prop;                  // [Q, N, 4] the proposed hands of the current move
    int32_t* anc;                    // [Q, N] ancestors of the current stage
    unsigned long long* accepted;    // [Q] accepted moves
    double* evidence;                // [Q]
    int32_t* resamples;              // [Q]
    double* acceptance;              // [Q]
    double* tr_loglik;               // trace (or NULL): [Q, K, N] l_k
    int32_t* tr_anc;                 // [Q, K, N] ancestor, -1 without a resample
    int32_t* tr_pairs;               // [Q, K, R] pair 0..2, -1 without a move
    uint8_t* tr_acc;                 // [Q, K, R, N]
    double* tr_prop;                 // [Q, K, R, N, 2] ell' of the pair's two seats
    float kappa;
    int32_t K, R;
};

// the pair of hidden seats of move mv at stage k (0: LHO + partner, 1: LHO + RHO, 2: partner + RHO), shared by the query
__device__ __forceinline__ int32_t smc_pair(uint64_t seed, int64_t g, int32_t k, int32_t mv) {
    const uint4 u = philox4x32(make_uint4((uint32_t)g, (uint32_t)((uint64_t)g >> 32), BRL_SMC_TAG + 128u * (uint32_t)k + 1u + (uint32_t)mv,
                                          0xFFFFFFFFu), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    return (int32_t)__umulhi(u.x, 3u);
}

__device__ __forceinline__ void pair_seats(int32_t pair, int32_t& r1, int32_t& r2) {
    r1 = pair == 2 ? 1 : 0;
    r2 = pair == 0 ? 1 : 2;
}

struct SmcWindow {  // the row set of stage k (move < 0) or of move `move` at stage k
    const uint8_t* flags;
    uint64_t seed;
    int64_t g0;
    int32_t k, move;
    __device__ __forceinline__ uint32_t seats(int64_t j, int32_t s) const {
        int32_t r1, r2;
        pair_seats(smc_pair(seed, g0 + j, k, move), r1, r2);
        return (1u << ((s + 1 + r1) & 3)) | (1u << ((s + 1 + r2) & 3));
    }
    __device__ __forceinline__ int32_t calls(int64_t j, int32_t s, int32_t sg, int32_t dealer, int32_t L) const {
        if (move < 0) return (flags[j] & kSmcLive) && k < L && ((dealer + k) & 3) == sg ? 1 : 0;
        if (!(flags[j] & kSmcMoved) || !((seats(j, s) >> sg) & 1u)) return 0;
        return calls_by(sg, dealer, min(L, k + 1));
    }
    __device__ __forceinline__ bool takes(int64_t j, int32_t s, int32_t c, int32_t sg) const {
        if (move < 0) return (flags[j] & kSmcLive) && c == k;
        return (flags[j] & kSmcMoved) && c <= k && ((seats(j, s) >> sg) & 1u);
    }
};

// l_k of particle i for every call of the window, in k order, added into lp[hidden seat] (0 LHO, 1 partner, 2 RHO)
__device__ __forceinline__ void smc_loglik(const PostArgs& a, const SmcWindow& w, int64_t j, int64_t i, double lp[3]) {
    const int32_t t = a.query[3 * j], s = a.query[3 * j + 1], L = a.query[3 * j + 2];
    const int32_t dealer = a.dealer ? (int32_t)(a.dealer[t] & 3) : 0;
    const int4 nv = reinterpret_cast<const int4*>(a.seat_nets)[j];
    const int32_t nets[4] = {nv.x, nv.y, nv.z, nv.w};
    int32_t seen[4] = {0, 0, 0, 0};
    const int32_t hi = min(L, w.k + 1);
    for (int32_t k = w.move < 0 ? w.k : 0; k < hi; ++k) {
        const int32_t sg = (dealer + k) & 3;
        if (sg == s || !w.takes(j, s, k, sg)) continue;
        const int32_t m = nets[sg];
        int al = 0;
        while (nets[al] != m) ++al;
        const int64_t rank = (int64_t)a.base[4 * j + sg] + seen[al]++;
        const PostSeg& d = a.seg[a.seg_prefix[m] + rank];
        const uint64_t legal = (uint64_t)d.legal_lo | ((uint64_t)d.legal_hi << 32);
        const float* l = a.logits + (a.group_off[m] + rank * a.N + i) * kNumActions;
        const float x = a.tau == 0.0f ? (post_argmax(l, legal) == d.call ? 0.0f : -INFINITY) : post_log_softmax(l, legal, d.call, a.tau);
        lp[(sg - s - 1) & 3] += (double)x;
    }
}

__global__ void __launch_bounds__(256) k_smc_init(const PostArgs a, const SmcArgs m) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.Q * a.N) return;
    const int64_t j = idx / a.N;
    a.logw[idx] = 0.0;
    m.ell[3 * idx] = m.ell[3 * idx + 1] = m.ell[3 * idx + 2] = 0.0;
    if (idx != j * a.N) return;
    if (a.status[j] == BRL_POST_OK && a.query[3 * j + 2] > m.K) a.status[j] = BRL_POST_STAGES;
    m.flags[j] = a.status[j] == BRL_POST_OK ? kSmcLive : 0;
    m.accepted[j] = 0ull;
    m.evidence[j] = 0.0;
    m.resamples[j] = 0;
    if (j == 0) a.meta[2] = 0;  // any layout of the call overflowed the capacity
}

// stage k's reweight: log w += l_k, ell[sigma_k] += l_k
__global__ void __launch_bounds__(256) k_smc_reweight(const PostArgs a, const SmcArgs m, int32_t k) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.Q * a.N) return;
    if (idx == 0 && a.meta[1]) a.meta[2] = 1;
    const int64_t j = idx / a.N, i = idx - j * a.N;
    const int32_t t = a.query[3 * j], s = a.query[3 * j + 1], L = a.query[3 * j + 2];
    const int32_t sg = ((a.dealer ? (int32_t)(a.dealer[t] & 3) : 0) + k) & 3;
    double l = __longlong_as_double(0x7FF8000000000000ll);
    if ((m.flags[j] & kSmcLive) && k < L && sg != s && !a.meta[1]) {
        double lp[3] = {0.0, 0.0, 0.0};
        smc_loglik(a, SmcWindow{m.flags, a.seed, a.g0, k, -1}, j, i, lp);
        const int r = (sg - s - 1) & 3;
        l = lp[r];
        a.logw[idx] += l;
        m.ell[3 * idx + r] += l;
    }
    if (m.tr_loglik) m.tr_loglik[(j * m.K + k) * a.N + i] = l;
}

// stage k's ESS test and systematic resampling: one thread per query, every sum in sample order
__global__ void __launch_bounds__(128) k_smc_resample(const PostArgs a, const SmcArgs m, int32_t k) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.Q) return;
    uint8_t f = m.flags[j] & kSmcLive;
    const int32_t t = a.query[3 * j], s = a.query[3 * j + 1], L = a.query[3 * j + 2];
    const int32_t sg = ((a.dealer ? (int32_t)(a.dealer[t] & 3) : 0) + k) & 3;
    if (f && k < L && sg != s) {
        const double* lw = a.logw + j * a.N;
        double mx = -INFINITY;
        for (int64_t i = 0; i < a.N; ++i) mx = fmax(mx, lw[i]);
        if (mx == -INFINITY) {
            f = 0;  // extinct
        } else {
            double W = 0.0, W2 = 0.0;
            for (int64_t i = 0; i < a.N; ++i) {
                const double w = exp(lw[i] - mx);
                W += w;
                W2 += w * w;
            }
            if (m.kappa >= 1.0f || W * W / W2 < (double)m.kappa * (double)a.N) {
                const uint4 u4 = philox4x32(make_uint4((uint32_t)(a.g0 + j), (uint32_t)((uint64_t)(a.g0 + j) >> 32),
                                                       BRL_SMC_TAG + 128u * (uint32_t)k, 0xFFFFFFFFu),
                                            make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32)));
                const double u = ((double)u4.x + 0.5) * 0x1p-32;
                int64_t n = 0;
                double C = exp(lw[0] - mx);
                for (int64_t i = 0; i < a.N; ++i) {
                    const double target = ((double)i + u) * W / (double)a.N;
                    while (C < target && n < a.N - 1) C += exp(lw[++n] - mx);
                    m.anc[j * a.N + i] = (int32_t)n;
                }
                m.evidence[j] += log(W / (double)a.N) + mx;
                m.resamples[j] += 1;
                f |= kSmcMoved;
            }
        }
    }
    m.flags[j] = f;
}

// copy each moved particle's hands and ell from its ancestor (into the tmp buffers, copied back by the host's memcpy)
__global__ void __launch_bounds__(256) k_smc_gather(const PostArgs a, const SmcArgs m, int32_t k) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.Q * a.N) return;
    const int64_t j = idx / a.N, i = idx - j * a.N;
    const bool moved = m.flags[j] & kSmcMoved;
    const int64_t src = moved ? j * a.N + m.anc[idx] : idx;
    const ulonglong2* h = reinterpret_cast<const ulonglong2*>(a.hands + 4 * src);
    ulonglong2* o = reinterpret_cast<ulonglong2*>(m.tmp_hands + 4 * idx);
    o[0] = h[0];
    o[1] = h[1];
    for (int r = 0; r < 3; ++r) m.tmp_ell[3 * idx + r] = m.ell[3 * src + r];
    if (moved) a.logw[idx] = 0.0;
    if (m.tr_anc) m.tr_anc[(j * m.K + k) * a.N + i] = moved ? m.anc[idx] : -1;
}

// move mv's proposal: swap a uniform card of r1 with a uniform card of r2 (the a-th / b-th set bit of the hand)
__device__ __forceinline__ int nth_card(uint64_t h, uint32_t n) {
    for (uint32_t x = 0; x < n; ++x) h &= h - 1;
    return __ffsll((long long)h) - 1;
}

__global__ void __launch_bounds__(256) k_smc_propose(const PostArgs a, const SmcArgs m, int32_t k, int32_t mv) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.Q * a.N) return;
    const int64_t j = idx / a.N, i = idx - j * a.N;
    if (!(m.flags[j] & kSmcMoved)) return;
    const int32_t s = a.query[3 * j + 1];
    int32_t r1, r2;
    pair_seats(smc_pair(a.seed, a.g0 + j, k, mv), r1, r2);
    const uint4 u = philox4x32(make_uint4((uint32_t)(a.g0 + j), (uint32_t)((uint64_t)(a.g0 + j) >> 32),
                                          BRL_SMC_TAG + 128u * (uint32_t)k + 1u + (uint32_t)mv, (uint32_t)i),
                               make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32)));
    uint64_t h[4];
    for (int x = 0; x < 4; ++x) h[x] = a.hands[4 * idx + x];
    const int s1 = (s + 1 + r1) & 3, s2 = (s + 1 + r2) & 3;
    const int c1 = nth_card(h[s1], __umulhi(u.x, 13u)), c2 = nth_card(h[s2], __umulhi(u.y, 13u));
    h[s1] ^= (1ull << c1) | (1ull << c2);
    h[s2] ^= (1ull << c1) | (1ull << c2);
    for (int x = 0; x < 4; ++x) m.prop[4 * idx + x] = h[x];
}

// move mv's Metropolis-Hastings test: accept iff log u < ell'[r1] + ell'[r2] - ell[r1] - ell[r2]
__global__ void __launch_bounds__(256) k_smc_accept(const PostArgs a, const SmcArgs m, int32_t k, int32_t mv) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.Q * a.N) return;
    if (idx == 0 && a.meta[1]) a.meta[2] = 1;
    const int64_t j = idx / a.N, i = idx - j * a.N;
    const bool moved = (m.flags[j] & kSmcMoved) && !a.meta[1];
    const int32_t pair = smc_pair(a.seed, a.g0 + j, k, mv);
    const int64_t tr = ((j * m.K + k) * m.R + mv) * a.N + i;
    if (m.tr_pairs && i == 0) m.tr_pairs[(j * m.K + k) * m.R + mv] = moved ? pair : -1;
    bool acc = false;
    double lp[3] = {0.0, 0.0, 0.0};
    int32_t r1, r2;
    pair_seats(pair, r1, r2);
    if (moved) {
        smc_loglik(a, SmcWindow{m.flags, a.seed, a.g0, k, mv}, j, i, lp);
        const uint4 u = philox4x32(make_uint4((uint32_t)(a.g0 + j), (uint32_t)((uint64_t)(a.g0 + j) >> 32),
                                              BRL_SMC_TAG + 128u * (uint32_t)k + 1u + (uint32_t)mv, (uint32_t)i),
                                   make_uint2((uint32_t)a.seed, (uint32_t)(a.seed >> 32)));
        const double delta = (lp[r1] + lp[r2]) - (m.ell[3 * idx + r1] + m.ell[3 * idx + r2]);
        acc = log(((double)u.z + 0.5) * 0x1p-32) < delta;
        if (acc) {
            for (int x = 0; x < 4; ++x) a.hands[4 * idx + x] = m.prop[4 * idx + x];
            m.ell[3 * idx + r1] = lp[r1];
            m.ell[3 * idx + r2] = lp[r2];
        }
        if (acc) atomicAdd(m.accepted + j, 1ull);
    }
    if (m.tr_acc) {
        m.tr_acc[tr] = acc;
        m.tr_prop[2 * tr] = moved ? lp[r1] : __longlong_as_double(0x7FF8000000000000ll);
        m.tr_prop[2 * tr + 1] = moved ? lp[r2] : __longlong_as_double(0x7FF8000000000000ll);
    }
}

// f18's NaN log w for queries without a posterior, and the sticky capacity flag for f18's reduction
__global__ void __launch_bounds__(256) k_smc_end(const PostArgs a, const SmcArgs m) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.Q * a.N) return;
    if (idx == 0) a.meta[1] = a.meta[2];
    const int64_t j = idx / a.N;
    if (a.status[j] != BRL_POST_OK || a.meta[2]) a.logw[idx] = __longlong_as_double(0x7FF8000000000000ll);
}

// the last factor of the evidence, the acceptance rate, NaN for queries without a posterior
__global__ void __launch_bounds__(128) k_smc_finish(const PostArgs a, const SmcArgs m) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.Q) return;
    const double nan = __longlong_as_double(0x7FF8000000000000ll);
    const double* wt = a.weights + 4 * j;
    const double proposed = (double)m.resamples[j] * m.R * a.N;
    if (a.status[j] != BRL_POST_OK) {
        m.evidence[j] = nan;
        m.acceptance[j] = nan;
        return;
    }
    m.evidence[j] = wt[3] == 0.0 ? -INFINITY : m.evidence[j] + (log(wt[1] / (double)a.N) + wt[0]);
    m.acceptance[j] = proposed > 0.0 ? (double)m.accepted[j] / proposed : nan;
}

// ---- scratch --------------------------------------------------------------------------------------------------------------
struct PostLayout {
    size_t meta, group_off, seg_prefix, totals, base, seg, rows, block_model, action, obs, logits, fwd, hands, logw, total;
};

static PostLayout post_layout(int64_t Q, int64_t N, int64_t cap, int64_t M) {
    PostLayout L{};
    size_t o = 0;
    auto take = [&](size_t bytes) {
        const size_t at = o;
        o += (bytes + 255) / 256 * 256;
        return at;
    };
    L.meta = take(16 * 4);
    L.group_off = take((size_t)(M + 1) * 8);
    L.seg_prefix = take((size_t)(M + 1) * 8);
    L.totals = take((size_t)M * 4);
    L.base = take((size_t)Q * 16);
    L.seg = take((size_t)(cap / N) * sizeof(PostSeg));
    L.rows = take((size_t)cap * 4);
    L.block_model = take((size_t)(cap / kGroupRows) * 4);
    L.action = take((size_t)cap * 4);
    L.obs = take((size_t)cap * kObsDim * 2);
    L.logits = take((size_t)cap * kNumActions * 4);
    L.fwd = take((size_t)brl_mlp_rows_scratch_bytes(cap));
    L.hands = take((size_t)(Q * N) * 32);
    L.logw = take((size_t)(Q * N) * 8);
    L.total = o;
    return L;
}


struct SmcLayout {
    PostLayout post;
    size_t ell, tmp_ell, tmp_hands, prop, anc, flags, accepted, total;
};

static SmcLayout smc_layout(int64_t Q, int64_t N, int64_t cap, int64_t M) {
    SmcLayout L{};
    L.post = post_layout(Q, N, cap, M);
    size_t o = L.post.total;
    auto take = [&](size_t bytes) {
        const size_t at = o;
        o += (bytes + 255) / 256 * 256;
        return at;
    };
    L.ell = take((size_t)(Q * N) * 24);
    L.tmp_ell = take((size_t)(Q * N) * 24);
    L.tmp_hands = take((size_t)(Q * N) * 32);
    L.prop = take((size_t)(Q * N) * 32);
    L.anc = take((size_t)(Q * N) * 4);
    L.flags = take((size_t)Q);
    L.accepted = take((size_t)Q * 8);
    L.total = o;
    return L;
}

// the parameter checks both ops share
static int32_t post_check(const char* who, const BrlParams& p) {
    const int64_t Q = p.n_envs, N = (int64_t)p.step, cap = p.state_stride, M = p.k_steps;
    const float tau = p.gamma;
    if (N < 1 || N > (1 << 24)) return fail(BRL_E_OPAQUE, "%s: step (samples per query) must be in [1, 2^24]", who);
    if (M <= 0) return fail(BRL_E_OPAQUE, "%s: k_steps (the pool's model count) must be > 0", who);
    if (cap < 0 || cap % kGroupRows != 0 || cap > ((int64_t)1 << 30))
        return fail(BRL_E_OPAQUE, "%s: state_stride (the row capacity) must be a multiple of %d in [0, 2^30]", who, kGroupRows);
    if (!(tau >= 0.0f) || tau == INFINITY) return fail(BRL_E_OPAQUE, "%s: gamma (the temperature) must be finite and >= 0", who);
    if (p.n_deals <= 0) return fail(BRL_E_OPAQUE, "%s: n_deals must be the number of deal-table rows (> 0)", who);
    if (Q > ((int64_t)1 << 31) / 4 || Q * N > ((int64_t)1 << 40)) return fail(BRL_E_OPAQUE, "%s: n_envs * step too large", who);
    if (p.flags & ~(BRL_F_MLP_BF16 | BRL_F_TUNE_MLP_LAYERS | BRL_F_TUNE_MLP_FUSED))
        return fail(BRL_E_OPAQUE, "%s: flags may hold BRL_F_MLP_BF16 and BRL_F_TUNE_MLP_* only", who);
    return BRL_OK;
}

// buffers [0]-[13] and the scratch of both ops; hands / logw: the caller's diagnostics, or NULL for scratch
static PostArgs post_args(void** b, const BrlParams& p, const PostLayout& L, uint64_t* hands, double* logw) {
    unsigned char* sc = static_cast<unsigned char*>(b[9]);
    PostArgs a{};
    a.table = static_cast<const uint8_t*>(b[0]);
    a.calls = static_cast<const uint8_t*>(b[1]);
    a.offsets = static_cast<const int64_t*>(b[2]);
    a.board = static_cast<const int32_t*>(b[3]);
    a.dealer = static_cast<const int8_t*>(b[4]);
    a.vul = static_cast<const uint8_t*>(b[5]);
    a.query = static_cast<const int32_t*>(b[6]);
    a.seat_nets = static_cast<const int32_t*>(b[7]);
    a.status = static_cast<int32_t*>(b[13]);
    a.meta = reinterpret_cast<int32_t*>(sc + L.meta);
    a.group_off = reinterpret_cast<int64_t*>(sc + L.group_off);
    a.seg_prefix = reinterpret_cast<int64_t*>(sc + L.seg_prefix);
    a.totals = reinterpret_cast<int32_t*>(sc + L.totals);
    a.base = reinterpret_cast<int32_t*>(sc + L.base);
    a.seg = reinterpret_cast<PostSeg*>(sc + L.seg);
    a.rows = reinterpret_cast<int32_t*>(sc + L.rows);
    a.block_model = reinterpret_cast<int32_t*>(sc + L.block_model);
    a.obs = sc + L.obs;
    a.logits = reinterpret_cast<const float*>(sc + L.logits);
    a.hands = hands ? hands : reinterpret_cast<uint64_t*>(sc + L.hands);
    a.logw = logw ? logw : reinterpret_cast<double*>(sc + L.logw);
    a.cards = static_cast<double*>(b[10]);
    a.features = static_cast<double*>(b[11]);
    a.weights = static_cast<double*>(b[12]);
    a.Q = p.n_envs;
    a.cap = p.state_stride;
    a.g0 = p.env_offset;
    a.seed = p.seed;
    a.N = (int32_t)p.step;
    a.M = (int32_t)p.k_steps;
    a.n_deals = p.n_deals;
    a.tau = p.gamma;
    return a;
}

// the grouped forward over the layout's rows, logits out
static int32_t post_forward(cudaStream_t s, const BrlParams& p, void** b, unsigned char* sc, const PostLayout& L, const PostArgs& a) {
    const int32_t fwd_flags = p.flags & (BRL_F_MLP_BF16 | BRL_F_TUNE_MLP_LAYERS | BRL_F_TUNE_MLP_FUSED);
    return launch_policy_grouped(s, fwd_flags, p.state_stride, p.k_steps, a.obs, static_cast<const unsigned char*>(b[8]), sc + L.fwd,
                                 nullptr, reinterpret_cast<int32_t*>(sc + L.action), a.rows, a.block_model, a.meta,
                                 reinterpret_cast<float*>(sc + L.logits));
}
}  // namespace brl

using namespace brl;

extern "C" {

int64_t brl_hand_posterior_scratch_bytes(int64_t n_queries, int64_t n_samples, int64_t row_capacity, int64_t n_models) {
    if (n_queries < 0 || n_samples <= 0 || row_capacity < 0 || n_models <= 0) return -1;
    return (int64_t)post_layout(n_queries, n_samples, row_capacity, n_models).total;
}

int32_t brl_hand_posterior(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    static const char* const who = "brl_hand_posterior";
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;
    if ((rc = post_check(who, *p))) return rc;
    static const char* const names[] = {"deal_table", "calls", "offsets", "board", "dealer", "vul", "query", "seat_nets", "pool",
                                        "scratch", "cards", "features", "weights", "status", "hands", "logw"};
    static const uint8_t align[] = {16, 1, 8, 4, 1, 1, 4, 16, 16, 16, 8, 8, 8, 4, 16, 8};
    const unsigned nullable = (1u << 3) | (1u << 4) | (1u << 5) | (1u << 14) | (1u << 15);
    if ((rc = check_buffers(who, b, names, 16, nullable, 0u, align))) return rc;
    if ((b[14] == nullptr) != (b[15] == nullptr)) return fail(BRL_E_BUFFER, "%s: buffers 'hands' and 'logw' go together", who);

    const int64_t Q = p->n_envs, N = (int64_t)p->step, cap = p->state_stride, M = p->k_steps;
    const PostLayout L = post_layout(Q, N, cap, M);
    unsigned char* sc = static_cast<unsigned char*>(b[9]);
    const PostArgs a = post_args(b, *p, L, static_cast<uint64_t*>(b[14]), static_cast<double*>(b[15]));

    if (cap > 0 && (rc = warm_policy_grouped(!(p->flags & BRL_F_MLP_BF16)))) return rc;
    const cudaStream_t s = (cudaStream_t)stream;
    const unsigned qn_blocks = (unsigned)((Q * N + 255) / 256);
    k_post_check<<<(unsigned)Q, 128, 0, s>>>(a);
    k_post_count<<<(unsigned)M, 1024, 0, s>>>(a);
    k_post_layout<<<1, 1, 0, s>>>(a);
    if (cap > 0) {
        k_post_rows<<<(unsigned)(cap / 256), 256, 0, s>>>(a);
        k_post_public<<<(unsigned)Q, 128, 0, s>>>(a);
    }
    k_post_sample<<<qn_blocks, 256, 0, s>>>(a);
    if (cap > 0) {
        k_post_expand<<<(unsigned)(cap / 8), 256, 0, s>>>(a);
        if ((rc = check_launch(who))) return rc;
        if ((rc = post_forward(s, *p, b, sc, L, a))) return rc;
    }
    k_post_loglik<<<qn_blocks, 256, 0, s>>>(a);
    k_post_reduce<<<(unsigned)Q, 512, 0, s>>>(a);
    return check_launch(who);
}

int64_t brl_hand_posterior_smc_scratch_bytes(int64_t n_queries, int64_t n_samples, int64_t row_capacity, int64_t n_models) {
    if (n_queries < 0 || n_samples <= 0 || row_capacity < 0 || n_models <= 0) return -1;
    return (int64_t)smc_layout(n_queries, n_samples, row_capacity, n_models).total;
}

int32_t brl_hand_posterior_smc(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    static const char* const who = "brl_hand_posterior_smc";
    if (opaque == nullptr || len != sizeof(BrlSmcParams))
        return fail(BRL_E_OPAQUE, "%s: opaque must be one BrlSmcParams (%zu bytes), got %zu", who, sizeof(BrlSmcParams), len);
    const BrlSmcParams* sp = static_cast<const BrlSmcParams*>(opaque);
    const BrlParams* p = &sp->post;
    if (p->n_envs < 0) return fail(BRL_E_OPAQUE, "%s: n_envs < 0", who);
    if (p->n_envs == 0) return BRL_OK;
    int32_t rc;
    if ((rc = post_check(who, *p))) return rc;
    if (!(sp->ess_threshold >= 0.0f && sp->ess_threshold <= 1.0f))
        return fail(BRL_E_OPAQUE, "%s: ess_threshold must be in [0, 1]", who);
    if (sp->moves < 0 || sp->moves > BRL_SMC_MAX_MOVES) return fail(BRL_E_OPAQUE, "%s: moves must be in [0, %d]", who, BRL_SMC_MAX_MOVES);
    if (sp->stages < 0 || sp->stages > BRL_SMC_MAX_STAGES)
        return fail(BRL_E_OPAQUE, "%s: stages must be in [0, %d]", who, BRL_SMC_MAX_STAGES);
    if (sp->reserved != 0) return fail(BRL_E_OPAQUE, "%s: reserved must be 0", who);
    static const char* const names[] = {"deal_table", "calls", "offsets", "board", "dealer", "vul", "query", "seat_nets", "pool",
                                        "scratch", "cards", "features", "weights", "status", "log_evidence", "resamples",
                                        "acceptance", "hands", "logw", "ell", "trace_loglik", "trace_ancestors", "trace_pairs",
                                        "trace_accepted", "trace_proposed"};
    static const uint8_t align[] = {16, 1, 8, 4, 1, 1, 4, 16, 16, 16, 8, 8, 8, 4, 8, 4, 8, 16, 8, 8, 8, 4, 4, 1, 8};
    const unsigned nullable = (1u << 3) | (1u << 4) | (1u << 5) | (0x1Fu << 17) | (0x1Fu << 20);
    // problems are reported in buffer order: the particle group [17..19] before the trace [20..24]
    if ((rc = check_buffers(who, b, names, 20, nullable, 0u, align))) return rc;
    if ((b[17] == nullptr) != (b[18] == nullptr) || (b[17] == nullptr) != (b[19] == nullptr))
        return fail(BRL_E_BUFFER, "%s: buffers 'hands', 'logw' and 'ell' go together", who);
    if ((rc = check_buffers(who, b, names, 25, nullable, 0u, align))) return rc;
    for (int k = 21; k < 25; ++k)
        if ((b[k] == nullptr) != (b[20] == nullptr)) return fail(BRL_E_BUFFER, "%s: the five trace buffers go together", who);

    const int64_t Q = p->n_envs, N = (int64_t)p->step, cap = p->state_stride, M = p->k_steps;
    const int32_t K = sp->stages, R = sp->moves;
    const SmcLayout L = smc_layout(Q, N, cap, M);
    unsigned char* sc = static_cast<unsigned char*>(b[9]);
    const PostArgs a = post_args(b, *p, L.post, static_cast<uint64_t*>(b[17]), static_cast<double*>(b[18]));
    SmcArgs m{};
    m.flags = sc + L.flags;
    m.ell = b[19] ? static_cast<double*>(b[19]) : reinterpret_cast<double*>(sc + L.ell);
    m.tmp_ell = reinterpret_cast<double*>(sc + L.tmp_ell);
    m.tmp_hands = reinterpret_cast<uint64_t*>(sc + L.tmp_hands);
    m.prop = reinterpret_cast<uint64_t*>(sc + L.prop);
    m.anc = reinterpret_cast<int32_t*>(sc + L.anc);
    m.accepted = reinterpret_cast<unsigned long long*>(sc + L.accepted);
    m.evidence = static_cast<double*>(b[14]);
    m.resamples = static_cast<int32_t*>(b[15]);
    m.acceptance = static_cast<double*>(b[16]);
    m.tr_loglik = static_cast<double*>(b[20]);
    m.tr_anc = static_cast<int32_t*>(b[21]);
    m.tr_pairs = static_cast<int32_t*>(b[22]);
    m.tr_acc = static_cast<uint8_t*>(b[23]);
    m.tr_prop = static_cast<double*>(b[24]);
    m.kappa = sp->ess_threshold;
    m.K = K;
    m.R = R;
    PostArgs moved = a;  // the move's forward reads the proposed hands
    moved.hands = m.prop;

    if (cap > 0 && (rc = warm_policy_grouped(!(p->flags & BRL_F_MLP_BF16)))) return rc;
    const cudaStream_t s = (cudaStream_t)stream;
    const unsigned qn_blocks = (unsigned)((Q * N + 255) / 256), q_blocks = (unsigned)((Q + 127) / 128);
    // one forward over the calls `rows` selects: the f18 layout, public pass, expansion and grouped forward
    auto forward = [&](const PostArgs& x, auto rows) -> int32_t {
        k_post_count<<<(unsigned)M, 1024, 0, s>>>(x, rows);
        k_post_layout<<<1, 1, 0, s>>>(x);
        if (cap == 0) return check_launch(who);
        k_post_rows<<<(unsigned)(cap / 256), 256, 0, s>>>(x);
        k_post_public<<<(unsigned)Q, 128, 0, s>>>(x, rows);
        k_post_expand<<<(unsigned)(cap / 8), 256, 0, s>>>(x);
        int32_t r = check_launch(who);
        return r ? r : post_forward(s, *p, b, sc, L.post, x);
    };
    k_post_check<<<(unsigned)Q, 128, 0, s>>>(a);
    k_post_sample<<<qn_blocks, 256, 0, s>>>(a);
    k_smc_init<<<qn_blocks, 256, 0, s>>>(a, m);
    for (int32_t k = 0; k < K; ++k) {
        SmcWindow w{m.flags, a.seed, a.g0, k, -1};
        if ((rc = forward(a, w))) return rc;
        k_smc_reweight<<<qn_blocks, 256, 0, s>>>(a, m, k);
        k_smc_resample<<<q_blocks, 128, 0, s>>>(a, m, k);
        k_smc_gather<<<qn_blocks, 256, 0, s>>>(a, m, k);
        cudaMemcpyAsync(a.hands, m.tmp_hands, (size_t)(Q * N) * 32, cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(m.ell, m.tmp_ell, (size_t)(Q * N) * 24, cudaMemcpyDeviceToDevice, s);
        for (int32_t mv = 0; mv < R; ++mv) {
            w.move = mv;
            k_smc_propose<<<qn_blocks, 256, 0, s>>>(a, m, k, mv);
            if ((rc = forward(moved, w))) return rc;
            k_smc_accept<<<qn_blocks, 256, 0, s>>>(a, m, k, mv);
        }
    }
    k_smc_end<<<qn_blocks, 256, 0, s>>>(a, m);
    k_post_reduce<<<(unsigned)Q, 512, 0, s>>>(a);
    k_smc_finish<<<q_blocks, 128, 0, s>>>(a, m);
    return check_launch(who);
}

}  // extern "C"
