// brl_algo.cu -- the small per-env algorithms around the environment: GAE reverse
// scan, masked categorical (mode / Gumbel-argmax sample / log-prob), IMP reward,
// match-statistic partial sums, transition reward gather, double-dummy par (its reward gather and match
// statistics), bidding-system histograms.  sm_100a only.
#include <math.h>

#include "common.h"
#include "env_device.cuh"

namespace brl {

static thread_local char g_last_error[512] = {0};
char* last_error_buffer() { return g_last_error; }

// ---- GAE -- src/gae.py:20-39 ---------------------------------------------------------------
// One thread per env walks T..0; every load/store is coalesced over the env axis
// ([T, n] time-major).  17 B per (t, env) of traffic; loads of a chunk are issued
// before the dependent chain so the scan is not latency-serialised per step.
// __fmul_rn/__fadd_rn keep the reference's operation order without FMA contraction.
constexpr int kGaeChunk = 8;

__global__ void __launch_bounds__(128) k_gae(const uint8_t* __restrict__ done, const float* __restrict__ value,
                                             const float* __restrict__ reward, const float* __restrict__ last_val,
                                             float* __restrict__ adv, float* __restrict__ targets, int T, int64_t n,
                                             float gamma, float lam) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float gae = 0.0f, next_value = last_val[i];
    const float gl = __fmul_rn(gamma, lam);
    for (int t0 = T; t0 > 0; t0 -= kGaeChunk) {
        float v[kGaeChunk], r[kGaeChunk];
        uint8_t d[kGaeChunk];
#pragma unroll
        for (int k = 0; k < kGaeChunk; ++k) {
            int t = t0 - 1 - k;
            if (t >= 0) {
                int64_t idx = (int64_t)t * n + i;
                v[k] = value[idx];
                r[k] = reward[idx];
                d[k] = done[idx];
            }
        }
#pragma unroll
        for (int k = 0; k < kGaeChunk; ++k) {
            int t = t0 - 1 - k;
            if (t >= 0) {
                int64_t idx = (int64_t)t * n + i;
                float nd = 1.0f - (float)d[k];
                float delta = __fadd_rn(__fadd_rn(r[k], __fmul_rn(__fmul_rn(gamma, next_value), nd)), -v[k]);
                gae = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, nd), gae));
                next_value = v[k];
                adv[idx] = gae;
                targets[idx] = __fadd_rn(gae, v[k]);
            }
        }
    }
}

// ---- masked categorical -- src/roll_out.py:27-30,79-81; src/evaluation.py:128-133 -----------
// where(mask, logits, -inf); mode = first argmax; sample = argmax(logits + Gumbel);
// log_prob = log_softmax(masked logits)[action].  One warp per env row.
__global__ void __launch_bounds__(128) k_categorical(const float* __restrict__ logits, const uint8_t* __restrict__ mask,
                                                     int32_t* __restrict__ action, float* __restrict__ log_prob,
                                                     int64_t n, int sample, uint64_t seed, int64_t env_offset,
                                                     uint32_t step, const int32_t* __restrict__ row_index,
                                                     float* __restrict__ logits_by_env) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n; r += n_warps) {
        // row_index: logits are compact ([n, 38] for the listed rows); mask / action / log_prob / RNG counter are by env
        const int64_t row = row_index ? (int64_t)row_index[r] : r;
        const float* l = logits + r * kNumActions;
        const uint8_t* m = mask ? mask + row * kNumActions : nullptr;
        float best = -INFINITY, mx = -INFINITY;
        int best_a = kNumActions;
        float lv[2];
        bool ok[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            int a = lane + 32 * k;
            ok[k] = a < kNumActions && (m == nullptr || m[a] != 0);
            if (logits_by_env && a < kNumActions) logits_by_env[row * kNumActions + a] = l[a];
            lv[k] = ok[k] ? l[a] : -INFINITY;
            if (ok[k]) {
                float v = lv[k];
                if (sample) {
                    uint64_t g = (uint64_t)(env_offset + row);
                    uint4 r = philox4x32(make_uint4((uint32_t)g, (uint32_t)(g >> 32), kTagGum + (uint32_t)(a >> 2), step),
                                         make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
                    uint32_t w = (a & 3) == 0 ? r.x : ((a & 3) == 1 ? r.y : ((a & 3) == 2 ? r.z : r.w));
                    float u = ((float)(w >> 8) + 0.5f) * (1.0f / 16777216.0f);
                    v += -logf(-logf(u));
                }
                if (v > best) { best = v; best_a = a; }  // k ascending: ties keep the lower index
                mx = fmaxf(mx, lv[k]);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            float ob = __shfl_xor_sync(0xffffffffu, best, o);
            int oa = __shfl_xor_sync(0xffffffffu, best_a, o);
            if (ob > best || (ob == best && oa < best_a)) { best = ob; best_a = oa; }
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        float se = 0.0f;
#pragma unroll
        for (int k = 0; k < 2; ++k)
            if (ok[k]) se += expf(lv[k] - mx);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
        if (best_a >= kNumActions) best_a = 0;  // no legal action: cannot happen for a valid mask
        float la = __shfl_sync(0xffffffffu, best_a >= 32 ? lv[1] : lv[0], best_a & 31);
        if (lane == 0) {
            if (action) action[row] = best_a;
            if (log_prob) log_prob[row] = la - mx - logf(se);
        }
    }
}

// ---- live-env compaction by acting team -- src/evaluation.py:124-151 ---------------------------
// The reference's vmapped loop runs BOTH teams' nets on every env every iteration and selects by
// `current_player < 2`, and keeps stepping finished envs until the slowest auction ends.  Here the envs still playing
// are listed per acting team (players 0/1 = team 1) so each net runs on exactly the rows it decides.  One block =
// 1024 consecutive envs: ballot + popc give every env its slot inside the block, one atomicAdd per block and team
// reserves the block's range (rows ascend within a block; block order is the order of arrival -- the consumers are
// row-order independent).
__global__ void __launch_bounds__(1024) k_team_rows(const int8_t* __restrict__ player, const uint8_t* __restrict__ done,
                                                    int32_t* __restrict__ rows1, int32_t* __restrict__ rows2,
                                                    int32_t* __restrict__ counts, int64_t n) {
    __shared__ int warp_cnt[2][32];
    __shared__ int base[2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * 1024 + threadIdx.x;
    const bool live = i < n && (done == nullptr || done[i] == 0);
    const bool t1 = live && player[i] < 2, t2 = live && !t1;
    const unsigned b1 = __ballot_sync(0xffffffffu, t1), b2 = __ballot_sync(0xffffffffu, t2);
    if (lane == 0) { warp_cnt[0][warp] = __popc(b1); warp_cnt[1][warp] = __popc(b2); }
    __syncthreads();
    if (warp < 2) {  // exclusive scan of the 32 warp counts of team `warp`
        const int c = warp_cnt[warp][lane];
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        warp_cnt[warp][lane] = incl - c;
        if (lane == 31) base[warp] = incl > 0 ? atomicAdd(&counts[warp], incl) : 0;
    }
    __syncthreads();
    const unsigned below = (1u << lane) - 1u;
    if (t1) rows1[base[0] + warp_cnt[0][warp] + __popc(b1 & below)] = (int32_t)i;
    if (t2) rows2[base[1] + warp_cnt[1][warp] + __popc(b2 & below)] = (int32_t)i;
}

// ---- live-env grouping by acting net over a pool (workspace/eval_selfplay_league.py) ---------------------------
// k_team_rows for many matches at once: env i is played by net env_models[i][0] for players 0/1 and env_models[i][1] for
// players 2/3 (src/evaluation.py:124-151); with BRL_F_PLAYER_MODELS (kStride 4) by net env_models[i][player] of each player.  Count per net, lay the nets' groups out padded to kGroupRows rows, scatter.  The
// envs of one match are contiguous, so a warp nearly always holds one or two nets: one atomic per net and warp.
// A live env whose acting net id is outside [0, M) invalidates the grouping: offsets[M] (the count the host reads anyway to
// size the forward) becomes -1, so the error surfaces before any forward runs, without an extra host read.
constexpr int kNotListed = -1, kBadModel = -2;
template <int kStride>
__device__ __forceinline__ int acting_model(int player, const int32_t* env_models, int64_t i, int n_models) {
    static_assert(kStride == 2 || kStride == 4, "env_models holds a net per team or per player");
    const int m = env_models[kStride * i + (kStride == 4 ? (player & 3) : (player < 2 ? 0 : 1))];
    return m >= 0 && m < n_models ? m : kBadModel;
}

template <int kStride>
__device__ __forceinline__ int acting_model(const int8_t* player, const uint8_t* done, const int32_t* env_models, int64_t i,
                                            int64_t n, int n_models) {
    if (i >= n || (done != nullptr && done[i] != 0)) return kNotListed;
    return acting_model<kStride>(player[i], env_models, i, n_models);
}

template <int kStride>
__global__ void __launch_bounds__(256) k_model_count(const int8_t* __restrict__ player, const uint8_t* __restrict__ done,
                                                     const int32_t* __restrict__ env_models, int32_t* __restrict__ counts,
                                                     int32_t* __restrict__ offsets, int64_t n, int n_models) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int m = acting_model<kStride>(player, done, env_models, i, n, n_models);
    const unsigned peers = __match_any_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) != __ffs(peers) - 1) return;
    if (m >= 0) atomicAdd(&counts[m], __popc(peers));
    else if (m == kBadModel) offsets[n_models] = -1;  // zeroed before this launch; read by k_model_offsets
}

// one block: offsets[m] = sum of the padded sizes of nets < m, offsets[M] = padded total (or -1 when k_model_count met a bad
// id); the block ids of each group, -1 in its padding rows; counts are reset to serve as the scatter's cursors (the scatter
// brings them back to the counts)
__global__ void __launch_bounds__(1024) k_model_offsets(int32_t* __restrict__ counts, int32_t* __restrict__ offsets,
                                                        int32_t* __restrict__ block_model, int32_t* __restrict__ rows, int n_models) {
    __shared__ int warp_sum[32];
    __shared__ int carry, bad;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        carry = 0;
        bad = offsets[n_models] < 0;
    }
    __syncthreads();
    for (int c0 = 0; c0 < n_models; c0 += 1024) {
        const int m = c0 + (int)threadIdx.x;
        const int padded = m < n_models ? (counts[m] + kGroupRows - 1) / kGroupRows * kGroupRows : 0;
        int incl = padded;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const int ws = warp_sum[lane];
            int wi = ws;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += v;
            }
            warp_sum[lane] = wi - ws;
        }
        __syncthreads();
        const int off = carry + warp_sum[warp] + incl - padded;
        if (m < n_models) {
            offsets[m] = off;
            const int cnt = counts[m];
            for (int r = off + cnt; r < off + padded; ++r) rows[r] = -1;
            for (int bl = off / kGroupRows; bl < (off + padded) / kGroupRows; ++bl) block_model[bl] = m;
            counts[m] = 0;
        }
        __syncthreads();
        if (threadIdx.x == 1023) carry = off + padded;
        __syncthreads();
    }
    if (threadIdx.x == 0) offsets[n_models] = bad ? -1 : carry;
}

template <int kStride>
__global__ void __launch_bounds__(256) k_model_scatter(const int8_t* __restrict__ player, const uint8_t* __restrict__ done,
                                                       const int32_t* __restrict__ env_models, const int32_t* __restrict__ offsets,
                                                       int32_t* __restrict__ cursor, int32_t* __restrict__ rows, int64_t n, int n_models) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int m = acting_model<kStride>(player, done, env_models, i, n, n_models);
    const unsigned peers = __match_any_sync(0xffffffffu, m);
    const int leader = __ffs(peers) - 1;
    int base = 0;
    if (m >= 0 && lane == leader) base = atomicAdd(&cursor[m], __popc(peers));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (m >= 0) rows[offsets[m] + base + __popc(peers & ((1u << lane) - 1u))] = (int32_t)i;
}

// ---- bidding-system statistics (env_device.cuh, DESIGN.md f15) ---------------------------------------------------------------
// One decision per live env, in the state before the step, into the histogram of the net acting there (acting_model, the rule
// of brl_model_rows; no env_models: net 0).  A call outside 0..37 or a net id outside [0, M) is not counted.
template <int kStride>
__global__ void __launch_bounds__(256) k_system_stats(const uint4* __restrict__ state, int64_t stride, const uint8_t* __restrict__ table,
                                                      const int32_t* __restrict__ action, const uint8_t* __restrict__ done,
                                                      const int32_t* __restrict__ env_models, uint32_t* __restrict__ hist, int64_t n,
                                                      int n_models) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || (done != nullptr && done[i] != 0)) return;
    const int32_t a = action[i];
    if (a < 0 || a >= kNumActions) return;
    Env e;
    load_env(state, stride, i, e);
    const uint32_t seat = f_cur_seat(e);
    const int m = env_models != nullptr ? acting_model<kStride>((int)f_player_at(e, seat), env_models, i, n_models) : 0;
    if (m < 0) return;
    system_count(hist + m * kSysCells, system_context(system_prefix(e)), (uint32_t)a, hand_features(TableRows{table}.hand(e.deal, seat)));
}

// Every call of stored auctions, one thread per auction: auction t is calls[offsets[t], offsets[t + 1]) on deal row board[t]
// (NULL: t) with dealer dealer[t] (NULL: North).  The calls and rows are the caller's checked input.
__global__ void __launch_bounds__(256) k_system_stats_auctions(const uint8_t* __restrict__ table, const uint8_t* __restrict__ calls,
                                                               const int64_t* __restrict__ offsets, const int32_t* __restrict__ board,
                                                               const int8_t* __restrict__ dealer, uint32_t* __restrict__ hist,
                                                               int64_t n) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint32_t row = board != nullptr ? (uint32_t)board[t] : (uint32_t)t;
    const uint32_t d = dealer != nullptr ? (uint32_t)dealer[t] & 3u : 0u;
    const TableRows rows{table};
    HandFeatures f[4];
#pragma unroll
    for (uint32_t s = 0; s < 4u; ++s) f[s] = hand_features(rows.hand(row, s));
    SystemPrefix p{};
    const int64_t end = offsets[t + 1];
    for (int64_t k = offsets[t]; k < end; ++k) {
        const uint32_t c = calls[k], seat = (d + p.t) & 3u;
        const HandFeatures& h = seat == 0u ? f[0] : (seat == 1u ? f[1] : (seat == 2u ? f[2] : f[3]));
        system_count(hist, system_context(p), c, h);
        system_push(p, c);
    }
}

// ---- _imp_reward -- src/duplicate.py:15-70 ----------------------------------------------------
__global__ void __launch_bounds__(256) k_imp_reward(const float4* __restrict__ a, const float4* __restrict__ b,
                                                    float4* __restrict__ out, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = imp_of_difference(a[i].x + b[i].x);
    out[i] = make_float4(s, s, -s, -s);
}

// ---- match statistics partial sums -- src/evaluation.py:199-201 -------------------------------
// sums[0..3] += {n, sum x, sum x^2, #(x > 0)} in double; the caller all-reduces the 8
// doubles across ranks (one NCCL all-reduce) and forms mean / SE(ddof=1) / win-rate.
__global__ void __launch_bounds__(256) k_match_stats(const float* __restrict__ x, double* __restrict__ sums, int64_t n) {
    double s1 = 0.0, s2 = 0.0, w = 0.0, c = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double v = (double)x[i];
        s1 += v;
        s2 += v * v;
        w += v > 0.0 ? 1.0 : 0.0;
        c += 1.0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        w += __shfl_xor_sync(0xffffffffu, w, o);
        c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    __shared__ double sh[4][8];
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { sh[0][warp] = c; sh[1][warp] = s1; sh[2][warp] = s2; sh[3][warp] = w; }
    __syncthreads();
    if (threadIdx.x < 4) {
        double t = 0.0;
        for (int k = 0; k < (int)(blockDim.x >> 5); ++k) t += sh[threadIdx.x][k];
        atomicAdd(&sums[threadIdx.x], t);
    }
}

// the same sums over P contiguous env ranges [offsets[p], offsets[p + 1]) into sums[p][0..3] (the matches of a league
// chunk); the grid's y dimension strides over the ranges, so P is not bounded by it.  The values are integer IMPs, so every
// entry equals k_match_stats on that slice exactly.
__global__ void __launch_bounds__(256) k_match_stats_ranges(const float* __restrict__ x, const int64_t* __restrict__ offsets,
                                                            double* __restrict__ sums, int64_t n_ranges) {
    __shared__ double sh[4][8];
    for (int64_t p = blockIdx.y; p < n_ranges; p += gridDim.y) {
        const int64_t lo = offsets[p], hi = offsets[p + 1];
        double s1 = 0.0, s2 = 0.0, w = 0.0, c = 0.0;
        for (int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (int64_t)gridDim.x * blockDim.x) {
            double v = (double)x[i];
            s1 += v;
            s2 += v * v;
            w += v > 0.0 ? 1.0 : 0.0;
            c += 1.0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            s2 += __shfl_xor_sync(0xffffffffu, s2, o);
            w += __shfl_xor_sync(0xffffffffu, w, o);
            c += __shfl_xor_sync(0xffffffffu, c, o);
        }
        int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (lane == 0) { sh[0][warp] = c; sh[1][warp] = s1; sh[2][warp] = s2; sh[3][warp] = w; }
        __syncthreads();
        if (threadIdx.x < 4) {
            double t = 0.0;
            for (int k = 0; k < (int)(blockDim.x >> 5); ++k) t += sh[threadIdx.x][k];
            if (t != 0.0) atomicAdd(&sums[8 * p + threadIdx.x], t);
        }
        __syncthreads();  // sh is reused by the next range
    }
}

// ---- roll_out bookkeeping -- src/roll_out.py:85-94: rewards[actor] / reward_scale -------------
// With `done` / `count`: also terminated_count += sum(done) (src/roll_out.py:85), one atomic per block.
__global__ void __launch_bounds__(256) k_gather_reward(const float* __restrict__ rewards, const int8_t* __restrict__ actor,
                                                       float* __restrict__ out, int64_t n, float scale,
                                                       const uint8_t* __restrict__ done, unsigned long long* __restrict__ count) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = rewards[4 * i + (actor[i] & 3)] / scale;
    if (count != nullptr) {
        const int c = __syncthreads_count(i < n && done[i] != 0);
        if (threadIdx.x == 0 && c > 0) atomicAdd(count, (unsigned long long)c);
    }
}

// ---- double-dummy par of each env's board (par_score), in the rewards layout by player id ------------------------------
// Only the A word (dealer, vulnerability, seating) and the deal index of the packed state are read.
__global__ void __launch_bounds__(256) k_par(const uint4* __restrict__ state, int64_t stride, const uint8_t* __restrict__ table,
                                             float4* __restrict__ par, int32_t* __restrict__ contract, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Env e;
    e.A = state[3 * stride + i].z;
    e.deal = state[4 * stride + i].w;
    const Par p = par_score(e, TableRows{table});
    const float v = (float)((f_player_at(e, 0u) >> 1) == 0u ? p.ns : -p.ns);  // par of the team of player ids {0, 1}
    par[i] = make_float4(v, v, -v, -v);
    if (contract != nullptr) contract[i] = p.contract;
}

// bidding against par over the two tables of a duplicate match, for the team of player ids {0, 1}: per table the IMPs of its
// score against par and whether its final contract is the par contract (level, strain and declaring side; doubles ignored;
// two passed-out boards match).  Table B has table A's board with the teams' seats swapped (env_duplicate_init), so its par
// by player id is table A's negated.  sums[0..4] += {tables, sum imp, sum imp^2, sum |imp|, #par contract} in double.
__device__ __forceinline__ bool reached_par(uint32_t seating, int32_t last_bid, int32_t last_bidder, int32_t par_contract) {
    if (last_bid < 0 || par_contract < 0) return last_bid < 0 && par_contract < 0;
    uint32_t side = 0u;  // the side of the seat the last bidder sits in
#pragma unroll
    for (uint32_t s = 0; s < 4u; ++s)
        if (((seating >> (2u * s)) & 3u) == (uint32_t)last_bidder) side = s & 1u;
    return last_bid == (par_contract & 0xFF) && side == ((uint32_t)par_contract >> 8 & 1u);
}

__global__ void __launch_bounds__(256) k_par_stats(const uint4* __restrict__ state, int64_t stride, const uint8_t* __restrict__ table,
                                                   const float* __restrict__ rew_a, const int32_t* __restrict__ bid_a,
                                                   const int32_t* __restrict__ bidder_a, const float* __restrict__ rew_b,
                                                   const int32_t* __restrict__ bid_b, const int32_t* __restrict__ bidder_b,
                                                   double* __restrict__ sums, int64_t n) {
    double acc[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        Env e;
        e.A = state[3 * stride + i].z;
        e.deal = state[4 * stride + i].w;
        const Par p = par_score(e, TableRows{table});
        const uint32_t s_a = f_seating(e);
        const uint32_t s_b = (s_a >> 2 & 3u) | (s_a & 3u) << 2 | (s_a >> 6 & 3u) << 4 | (s_a >> 4 & 3u) << 6;  // env_duplicate_init
        const float par_a = (float)((s_a & 3u) >> 1 == 0u ? p.ns : -p.ns);  // par of player ids {0, 1} at table A
        const float imp_a = imp_of_difference(rew_a[4 * i] - par_a), imp_b = imp_of_difference(rew_b[4 * i] + par_a);
        acc[0] += 2.0;
        acc[1] += (double)imp_a + (double)imp_b;
        acc[2] += (double)imp_a * imp_a + (double)imp_b * imp_b;
        acc[3] += (double)fabsf(imp_a) + (double)fabsf(imp_b);
        acc[4] += (reached_par(s_a, bid_a[i], bidder_a[i], p.contract) ? 1.0 : 0.0) +
                  (reached_par(s_b, bid_b[i], bidder_b[i], p.contract) ? 1.0 : 0.0);
    }
    __shared__ double sh[5][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
        if (lane == 0) sh[k][warp] = acc[k];
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        double t = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sh[threadIdx.x][w];
        if (t != 0.0) atomicAdd(&sums[threadIdx.x], t);
    }
}

// k_gather_reward's par counterpart: a finished board's reward is IMP(score - par) / 24 from the actor's side
__global__ void __launch_bounds__(256) k_gather_reward_par(const float* __restrict__ rewards, const int8_t* __restrict__ actor,
                                                           const float* __restrict__ par, const uint8_t* __restrict__ done,
                                                           float* __restrict__ out, int64_t n,
                                                           unsigned long long* __restrict__ count) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool d = i < n && done[i] != 0;
    if (i < n) {
        const int64_t k = 4 * i + (actor[i] & 3);
        out[i] = d ? imp_of_difference(rewards[k] - par[k]) / 24.0f : 0.0f;
    }
    if (count != nullptr) {
        const int c = __syncthreads_count(d);
        if (threadIdx.x == 0 && c > 0) atomicAdd(count, (unsigned long long)c);
    }
}


// brl_model_rows' three kernels for env_models[n, kStride] (counts and offsets[M] already zeroed)
template <int kStride>
static void model_rows_launch(cudaStream_t s, void** b, int64_t n, int n_models) {
    const unsigned grid = (unsigned)((n + 255) / 256);
    const int8_t* player = static_cast<const int8_t*>(b[0]);
    const uint8_t* done = static_cast<const uint8_t*>(b[1]);
    const int32_t* env_models = static_cast<const int32_t*>(b[2]);
    int32_t* counts = static_cast<int32_t*>(b[4]);
    k_model_count<kStride><<<grid, 256, 0, s>>>(player, done, env_models, counts, static_cast<int32_t*>(b[5]), n, n_models);
    k_model_offsets<<<1, 1024, 0, s>>>(counts, static_cast<int32_t*>(b[5]), static_cast<int32_t*>(b[6]), static_cast<int32_t*>(b[3]),
                                       n_models);
    k_model_scatter<kStride><<<grid, 256, 0, s>>>(player, done, env_models, static_cast<const int32_t*>(b[5]), counts,
                                                  static_cast<int32_t*>(b[3]), n, n_models);
}

int32_t launch_categorical(cudaStream_t stream, const float* logits, const unsigned char* mask, int32_t* action, float* log_prob,
                           int64_t n, int sample, uint64_t seed, int64_t env_offset, uint32_t step, const int32_t* row_index, float* logits_by_env) {
    unsigned grid = (unsigned)((n + 3) / 4);  // one warp per env row
    if (grid > 148u * 16u) grid = 148u * 16u;
    k_categorical<<<grid, 128, 0, stream>>>(logits, mask, action, log_prob, n, sample, seed, env_offset, step, row_index, logits_by_env);
    return check_launch("brl_categorical");
}

}  // namespace brl

using namespace brl;

extern "C" {

const char* brl_last_error(void) { return last_error_buffer(); }
int32_t brl_abi_version(void) { return BRL_ABI_VERSION; }

int32_t brl_gae(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    static const char* names[] = {"done", "value", "reward", "last_val", "advantages", "targets"};
    for (int k = 0; k < 6; ++k)
        if (b[k] == nullptr) return fail(BRL_E_BUFFER, "brl_gae: buffer '%s' is NULL", names[k]);
    if (p->k_steps <= 0) return fail(BRL_E_OPAQUE, "brl_gae: k_steps (T) must be > 0");
    k_gae<<<(unsigned)((p->n_envs + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        static_cast<const uint8_t*>(b[0]), static_cast<const float*>(b[1]), static_cast<const float*>(b[2]),
        static_cast<const float*>(b[3]), static_cast<float*>(b[4]), static_cast<float*>(b[5]), p->k_steps, p->n_envs,
        p->gamma, p->gae_lambda);
    return check_launch("brl_gae");
}

int32_t brl_categorical(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    if (b[0] == nullptr) return fail(BRL_E_BUFFER, "brl_categorical: buffer 'logits' is NULL");
    return launch_categorical((cudaStream_t)stream, static_cast<const float*>(b[0]), static_cast<const uint8_t*>(b[1]),
                              static_cast<int32_t*>(b[2]), static_cast<float*>(b[3]), p->n_envs,
                              (p->flags & BRL_F_SAMPLE) ? 1 : 0, p->seed, p->env_offset, p->step, nullptr);
}

int32_t brl_team_rows(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) {  // an empty batch: both lists are empty
        if (b[4] != nullptr) cudaMemsetAsync(b[4], 0, 2 * sizeof(int32_t), (cudaStream_t)stream);
        return check_launch("brl_team_rows");
    }
    BRL_REQUIRE(b[0], "current_player");
    BRL_REQUIRE(b[2], "rows_team1");
    BRL_REQUIRE(b[3], "rows_team2");
    BRL_REQUIRE(b[4], "counts");
    if (cudaMemsetAsync(b[4], 0, 2 * sizeof(int32_t), (cudaStream_t)stream) != cudaSuccess) return check_launch("brl_team_rows");
    unsigned grid = (unsigned)((p->n_envs + 1023) / 1024);
    k_team_rows<<<grid, 1024, 0, (cudaStream_t)stream>>>(static_cast<const int8_t*>(b[0]), static_cast<const uint8_t*>(b[1]),
                                                         static_cast<int32_t*>(b[2]), static_cast<int32_t*>(b[3]),
                                                         static_cast<int32_t*>(b[4]), p->n_envs);
    return check_launch("brl_team_rows");
}

int32_t brl_imp_reward(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "a_rewards");
    BRL_REQUIRE(b[1], "b_rewards");
    BRL_REQUIRE(b[2], "imp");
    k_imp_reward<<<(unsigned)((p->n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        static_cast<const float4*>(b[0]), static_cast<const float4*>(b[1]), static_cast<float4*>(b[2]), p->n_envs);
    return check_launch("brl_imp_reward");
}

int32_t brl_match_stats(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    if (b[0] == nullptr || b[1] == nullptr) return fail(BRL_E_BUFFER, "brl_match_stats: NULL buffer");
    unsigned grid = (unsigned)((p->n_envs + 255) / 256);
    if (grid > 148u * 4u) grid = 148u * 4u;
    k_match_stats<<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const float*>(b[0]), static_cast<double*>(b[1]),
                                                          p->n_envs);
    return check_launch("brl_match_stats");
}

int32_t brl_match_stats_ranges(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // no ranges: a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "x");
    BRL_REQUIRE(b[1], "offsets");
    BRL_REQUIRE(b[2], "sums");
    const unsigned grid_y = (unsigned)(p->n_envs < 65535 ? p->n_envs : 65535);  // the kernel strides over the rest
    k_match_stats_ranges<<<dim3(4u, grid_y), 256, 0, (cudaStream_t)stream>>>(
        static_cast<const float*>(b[0]), static_cast<const int64_t*>(b[1]), static_cast<double*>(b[2]), p->n_envs);
    return check_launch("brl_match_stats_ranges");
}

int32_t brl_model_rows(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    const int64_t n_models = p->k_steps;
    if (n_models <= 0) return fail(BRL_E_OPAQUE, "brl_model_rows: k_steps (the pool's model count) must be > 0");
    cudaStream_t s = (cudaStream_t)stream;
    if (p->n_envs == 0) {  // an empty batch: every group is empty
        if (b[4] != nullptr) cudaMemsetAsync(b[4], 0, n_models * sizeof(int32_t), s);
        if (b[5] != nullptr) cudaMemsetAsync(b[5], 0, (n_models + 1) * sizeof(int32_t), s);
        return check_launch("brl_model_rows");
    }
    BRL_REQUIRE(b[0], "current_player");
    BRL_REQUIRE(b[2], "env_models");
    BRL_REQUIRE(b[3], "rows");
    BRL_REQUIRE(b[4], "counts");
    BRL_REQUIRE(b[5], "offsets");
    BRL_REQUIRE(b[6], "block_model");
    if (p->n_envs > INT32_MAX / 2) return fail(BRL_E_OPAQUE, "brl_model_rows: n_envs too large");
    int32_t* counts = static_cast<int32_t*>(b[4]);
    if (cudaMemsetAsync(counts, 0, n_models * sizeof(int32_t), s) != cudaSuccess ||
        cudaMemsetAsync(static_cast<int32_t*>(b[5]) + n_models, 0, sizeof(int32_t), s) != cudaSuccess)
        return check_launch("brl_model_rows");
    if (p->flags & BRL_F_PLAYER_MODELS)
        model_rows_launch<4>(s, b, p->n_envs, (int)n_models);
    else
        model_rows_launch<2>(s, b, p->n_envs, (int)n_models);
    return check_launch("brl_model_rows");
}

int32_t brl_gather_reward(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    if (b[0] == nullptr || b[1] == nullptr || b[2] == nullptr) return fail(BRL_E_BUFFER, "brl_gather_reward: NULL buffer");
    const bool counting = (p->flags & BRL_F_COUNT_DONE) != 0;
    if (counting && (b[3] == nullptr || b[4] == nullptr || (reinterpret_cast<uintptr_t>(b[4]) & 7u)))
        return fail(BRL_E_BUFFER, "brl_gather_reward: BRL_F_COUNT_DONE needs buffers [3] done and [4] count (8-byte aligned)");
    k_gather_reward<<<(unsigned)((p->n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        static_cast<const float*>(b[0]), static_cast<const int8_t*>(b[1]), static_cast<float*>(b[2]), p->n_envs,
        p->gamma, counting ? static_cast<const uint8_t*>(b[3]) : nullptr,
        counting ? static_cast<unsigned long long*>(b[4]) : nullptr);
    return check_launch("brl_gather_reward");
}

int32_t brl_par(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    static const char* names[] = {"state", "deal_table", "par", "contract"};
    if ((rc = check_buffers("brl_par", b, names, 4, 1u << 3, 1u << 0 | 1u << 2)) != BRL_OK) return rc;
    if ((reinterpret_cast<uintptr_t>(b[3]) & 3u) != 0) return fail(BRL_E_BUFFER, "brl_par: buffer 'contract' is not 4-byte aligned");
    const int64_t stride = p->state_stride > 0 ? p->state_stride : p->n_envs;
    if (stride < p->n_envs) return fail(BRL_E_OPAQUE, "brl_par: state_stride < n_envs");
    k_par<<<(unsigned)((p->n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        static_cast<const uint4*>(b[0]), stride, static_cast<const uint8_t*>(b[1]), static_cast<float4*>(b[2]),
        static_cast<int32_t*>(b[3]), p->n_envs);
    return check_launch("brl_par");
}

int32_t brl_gather_reward_par(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    static const char* names[] = {"rewards", "actor", "par", "done", "reward", "count"};
    const bool counting = (p->flags & BRL_F_COUNT_DONE) != 0;
    if ((rc = check_buffers("brl_gather_reward_par", b, names, 6, counting ? 0u : 1u << 5, 1u << 0 | 1u << 2)) != BRL_OK) return rc;
    if (counting && (reinterpret_cast<uintptr_t>(b[5]) & 7u) != 0)
        return fail(BRL_E_BUFFER, "brl_gather_reward_par: buffer 'count' is not 8-byte aligned");
    k_gather_reward_par<<<(unsigned)((p->n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        static_cast<const float*>(b[0]), static_cast<const int8_t*>(b[1]), static_cast<const float*>(b[2]),
        static_cast<const uint8_t*>(b[3]), static_cast<float*>(b[4]), p->n_envs,
        counting ? static_cast<unsigned long long*>(b[5]) : nullptr);
    return check_launch("brl_gather_reward_par");
}

int32_t brl_par_stats(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    static const char* names[] = {"state", "deal_table", "rewards_a", "last_bid_a", "last_bidder_a", "rewards_b", "last_bid_b",
                                  "last_bidder_b", "sums"};
    if ((rc = check_buffers("brl_par_stats", b, names, 9, 0u, 1u << 0 | 1u << 2 | 1u << 5 | 1u << 8)) != BRL_OK) return rc;
    const int64_t stride = p->state_stride > 0 ? p->state_stride : p->n_envs;
    if (stride < p->n_envs) return fail(BRL_E_OPAQUE, "brl_par_stats: state_stride < n_envs");
    unsigned grid = (unsigned)((p->n_envs + 255) / 256);
    if (grid > 148u * 4u) grid = 148u * 4u;
    k_par_stats<<<grid, 256, 0, (cudaStream_t)stream>>>(
        static_cast<const uint4*>(b[0]), stride, static_cast<const uint8_t*>(b[1]), static_cast<const float*>(b[2]),
        static_cast<const int32_t*>(b[3]), static_cast<const int32_t*>(b[4]), static_cast<const float*>(b[5]),
        static_cast<const int32_t*>(b[6]), static_cast<const int32_t*>(b[7]), static_cast<double*>(b[8]), p->n_envs);
    return check_launch("brl_par_stats");
}

int32_t brl_system_stats(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    if (p->k_steps <= 0) return fail(BRL_E_OPAQUE, "brl_system_stats: k_steps (the histogram's net count) must be > 0");
    static const char* names[] = {"state", "deal_table", "action", "done", "env_models", "hist"};
    if ((rc = check_buffers("brl_system_stats", b, names, 6, 1u << 3 | 1u << 4, 1u << 0)) != BRL_OK) return rc;
    const bool player_models = (p->flags & BRL_F_PLAYER_MODELS) != 0;
    if (player_models && b[4] == nullptr) return fail(BRL_E_BUFFER, "brl_system_stats: BRL_F_PLAYER_MODELS needs env_models [4] (i32[n, 4])");
    if ((reinterpret_cast<uintptr_t>(b[2]) | reinterpret_cast<uintptr_t>(b[4]) | reinterpret_cast<uintptr_t>(b[5])) & 3u)
        return fail(BRL_E_BUFFER, "brl_system_stats: action, env_models and hist must be 4-byte aligned");
    const int64_t stride = p->state_stride > 0 ? p->state_stride : p->n_envs;
    if (stride < p->n_envs) return fail(BRL_E_OPAQUE, "brl_system_stats: state_stride < n_envs");
    const unsigned grid = (unsigned)((p->n_envs + 255) / 256);
    const uint4* state = static_cast<const uint4*>(b[0]);
    const uint8_t* table = static_cast<const uint8_t*>(b[1]);
    const int32_t* action = static_cast<const int32_t*>(b[2]);
    const uint8_t* done = static_cast<const uint8_t*>(b[3]);
    const int32_t* env_models = static_cast<const int32_t*>(b[4]);
    uint32_t* hist = static_cast<uint32_t*>(b[5]);
    if (player_models)
        k_system_stats<4><<<grid, 256, 0, (cudaStream_t)stream>>>(state, stride, table, action, done, env_models, hist, p->n_envs,
                                                                 p->k_steps);
    else
        k_system_stats<2><<<grid, 256, 0, (cudaStream_t)stream>>>(state, stride, table, action, done, env_models, hist, p->n_envs,
                                                                 p->k_steps);
    return check_launch("brl_system_stats");
}

int32_t brl_system_stats_auctions(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // no auctions: a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    static const char* names[] = {"deal_table", "calls", "offsets", "board", "dealer", "hist"};
    if ((rc = check_buffers("brl_system_stats_auctions", b, names, 6, 1u << 3 | 1u << 4, 1u << 0)) != BRL_OK) return rc;
    if ((reinterpret_cast<uintptr_t>(b[2]) & 7u) || ((reinterpret_cast<uintptr_t>(b[3]) | reinterpret_cast<uintptr_t>(b[5])) & 3u))
        return fail(BRL_E_BUFFER, "brl_system_stats_auctions: offsets must be 8-byte aligned, board and hist 4-byte aligned");
    k_system_stats_auctions<<<(unsigned)((p->n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        static_cast<const uint8_t*>(b[0]), static_cast<const uint8_t*>(b[1]), static_cast<const int64_t*>(b[2]),
        static_cast<const int32_t*>(b[3]), static_cast<const int8_t*>(b[4]), static_cast<uint32_t*>(b[5]), p->n_envs);
    return check_launch("brl_system_stats_auctions");
}

}  // extern "C"
