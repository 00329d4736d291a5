// brl_posterior.cu -- hand reading (DESIGN.md f18, restated by tests/posterior_ref.py): the hidden hands an auction implies
// under the nets' own policies, by self-normalised importance sampling of the 39 cards the observer cannot see.
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

__global__ void __launch_bounds__(1024) k_post_count(const PostArgs a) {
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
                if (sg != s && n4[sg] == m) cnt += calls_by(sg, dealer, L);
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
__global__ void __launch_bounds__(128) k_post_public(const PostArgs a) {
    const int64_t j = blockIdx.x;
    if (a.status[j] != BRL_POST_OK || a.meta[1]) return;
    const PostQuery q = post_query(a, j);
    const int4 nv = reinterpret_cast<const int4*>(a.seat_nets)[j];
    const int32_t nets[4] = {nv.x, nv.y, nv.z, nv.w};
    for (int32_t k = threadIdx.x; k < q.L; k += blockDim.x) {
        const int32_t sg = (q.dealer + k) & 3;
        if (sg == q.s) continue;
        const int32_t m = nets[sg];
        int32_t rank = 0;  // earlier segments of this query in net m's group
        for (int32_t c = 0; c < k; ++c) {
            const int32_t sc = (q.dealer + c) & 3;
            rank += sc != q.s && nets[sc] == m;
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
    const int64_t Q = p->n_envs, N = (int64_t)p->step, cap = p->state_stride, M = p->k_steps;
    const float tau = p->gamma;
    if (N < 1 || N > (1 << 24)) return fail(BRL_E_OPAQUE, "%s: step (samples per query) must be in [1, 2^24]", who);
    if (M <= 0) return fail(BRL_E_OPAQUE, "%s: k_steps (the pool's model count) must be > 0", who);
    if (cap < 0 || cap % kGroupRows != 0 || cap > ((int64_t)1 << 30))
        return fail(BRL_E_OPAQUE, "%s: state_stride (the row capacity) must be a multiple of %d in [0, 2^30]", who, kGroupRows);
    if (!(tau >= 0.0f) || tau == INFINITY) return fail(BRL_E_OPAQUE, "%s: gamma (the temperature) must be finite and >= 0", who);
    if (p->n_deals <= 0) return fail(BRL_E_OPAQUE, "%s: n_deals must be the number of deal-table rows (> 0)", who);
    if (Q > ((int64_t)1 << 31) / 4 || Q * N > ((int64_t)1 << 40)) return fail(BRL_E_OPAQUE, "%s: n_envs * step too large", who);
    if (p->flags & ~(BRL_F_MLP_BF16 | BRL_F_TUNE_MLP_LAYERS | BRL_F_TUNE_MLP_FUSED))
        return fail(BRL_E_OPAQUE, "%s: flags may hold BRL_F_MLP_BF16 and BRL_F_TUNE_MLP_* only", who);
    static const char* const names[] = {"deal_table", "calls", "offsets", "board", "dealer", "vul", "query", "seat_nets", "pool",
                                        "scratch", "cards", "features", "weights", "status", "hands", "logw"};
    static const uint8_t align[] = {16, 1, 8, 4, 1, 1, 4, 16, 16, 16, 8, 8, 8, 4, 16, 8};
    const unsigned nullable = (1u << 3) | (1u << 4) | (1u << 5) | (1u << 14) | (1u << 15);
    if ((rc = check_buffers(who, b, names, 16, nullable, 0u, align))) return rc;
    if ((b[14] == nullptr) != (b[15] == nullptr)) return fail(BRL_E_BUFFER, "%s: buffers 'hands' and 'logw' go together", who);

    const PostLayout L = post_layout(Q, N, cap, M);
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
    a.hands = b[14] ? static_cast<uint64_t*>(b[14]) : reinterpret_cast<uint64_t*>(sc + L.hands);
    a.logw = b[15] ? static_cast<double*>(b[15]) : reinterpret_cast<double*>(sc + L.logw);
    a.cards = static_cast<double*>(b[10]);
    a.features = static_cast<double*>(b[11]);
    a.weights = static_cast<double*>(b[12]);
    a.Q = Q;
    a.cap = cap;
    a.g0 = p->env_offset;
    a.seed = p->seed;
    a.N = (int32_t)N;
    a.M = (int32_t)M;
    a.n_deals = p->n_deals;
    a.tau = tau;

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
        const int32_t fwd_flags = p->flags & (BRL_F_MLP_BF16 | BRL_F_TUNE_MLP_LAYERS | BRL_F_TUNE_MLP_FUSED);
        if ((rc = launch_policy_grouped(s, fwd_flags, cap, (int)M, a.obs, static_cast<const unsigned char*>(b[8]), sc + L.fwd, nullptr,
                                        reinterpret_cast<int32_t*>(sc + L.action), a.rows, a.block_model, a.meta,
                                        reinterpret_cast<float*>(sc + L.logits))))
            return rc;
    }
    k_post_loglik<<<qn_blocks, 256, 0, s>>>(a);
    k_post_reduce<<<(unsigned)Q, 512, 0, s>>>(a);
    return check_launch(who);
}

}  // extern "C"
