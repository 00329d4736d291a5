// brl_env.cu -- environment kernels (init / step / duplicate / rollout / observe /
// legal mask) and their C-ABI entry points.  sm_100a only.
//
// Execution model (DESIGN.md "Kernels"): a warp owns a tile of EPW consecutive envs.
//   phase 1  lanes 0..EPW-1: one env per lane -- load 80 B of packed state (5
//            coalesced 128-bit plane loads), apply the call, resolve a terminal
//            contract from the L2-resident deal table, auto-reset, and leave the
//            observation as 15 words of bits + the 38-bit legal mask in shared
//            memory; per-env scalars (rewards float4, terminated, current_player)
//            are stored directly.
//   phase 2  all 32 lanes: for every env of the tile expand the 480 observation bits
//            into one 1920-byte row with 128-bit coalesced stores (lane l writes
//            float4 l, l+32, l+64, l+96), and the tile's EPW*38 mask bytes as one
//            contiguous run of 128-bit stores.
// The HBM traffic is the outputs (1980 B per env-step) + 2 x 80 B of state; nothing
// is re-read.  EPW (8/16/32) trades phase-1 lane utilisation for more warps in
// flight at small env counts.
#include <cuda_bf16.h>

#include "common.h"
#include "env_device.cuh"
#include "obs_row.cuh"

namespace brl {

constexpr int kRowStride = 17;  // odd stride: conflict-free phase-1 writes

template <int EPW>
struct alignas(16) WarpTile {
    uint32_t R[EPW * kRowStride];
    uint64_t M[EPW + 2];
};

struct TableInfo {  // src/duplicate.py:138-144 as SoA
    uint8_t* terminated;
    float4* rewards;
    int32_t* last_bid;
    int32_t* last_bidder;
    uint8_t* call_x;
    uint8_t* call_xx;
};

struct EnvArgs {
    const uint4* state_in;
    uint4* state_out;
    const uint8_t* table;
    const int32_t* action;
    // outputs (per step; rollout advances them by n rows per step)
    void* obs;
    uint8_t* mask;
    float4* rewards;
    uint8_t* terminated;
    int8_t* current_player;
    int32_t* action_out;
    unsigned long long* stats;
    const uint32_t* uniforms;  // rollout: caller-supplied u32[K, n] action uniforms (NULL -> Philox)
    int16_t* result16;         // rollout: compact result i16[K, n] = 2 * rewards[player 0] + terminated (BRL_F_RESULT_I16)
    int uniform16;             // rollout: `uniforms` is u16[K, n] (BRL_F_UNIFORM_U16); u32 uniform = u16 << 16
    // produce-kernel inputs
    const uint64_t* keys;
    const int32_t* in_deal;
    const int32_t* in_dealer;
    const uint8_t* in_vul_ns;
    const uint8_t* in_vul_ew;
    const int8_t* in_players;
    const uint64_t* in_rng_key;
    const int8_t* in_player_id;
    TableInfo ta, tb;
    int64_t n, stride, env_offset;
    uint64_t seed;
    uint32_t n_deals, step;
    int32_t flags, k_steps, mode;
    float illegal_penalty, illegal_bonus;
    int mask_vec;  // mask rows may be written with 128-bit stores
    int balanced;  // warp-specialised rollout: envs split evenly over a grid that is a multiple of the SM count
};

// `nthreads` threads (this one is `tid`) write the nbytes = n_valid*38 mask bytes of a
// tile as one contiguous run; M[e] holds env e's 38 mask bits, M[n_valid] must be 0.
__device__ __forceinline__ void emit_mask_run(const uint64_t* M, int tid, int nthreads, uint8_t* base, int nbytes,
                                              int mask_vec) {
    if (mask_vec == 2) {
        // run starting at an arbitrary byte address (balanced env split): byte stores up to the first
        // 16-byte boundary, 128-bit stores for the body, byte stores for the tail
        const int head = (int)((16u - (uint32_t)(reinterpret_cast<uintptr_t>(base) & 15u)) & 15u);
        const int body_end = head + ((nbytes - head) > 0 ? ((nbytes - head) & ~15) : 0);
        for (int o = tid; o < nbytes; o += nthreads) {
            if (o >= head && o < body_end) continue;
            int e0 = o / kNumActions, a0 = o - e0 * kNumActions;
            base[o] = (uint8_t)((M[e0] >> a0) & 1ull);
        }
        for (int o = head + tid * 16; o < body_end; o += nthreads * 16) {
            int e0 = o / kNumActions, a0 = o - e0 * kNumActions;
            uint64_t bits = (M[e0] >> a0) | (M[e0 + 1] << (kNumActions - a0));
            uint32_t h = (uint32_t)bits & 0xFFFFu;
            *reinterpret_cast<uint4*>(base + o) =
                make_uint4(spread4(h & 15u), spread4((h >> 4) & 15u), spread4((h >> 8) & 15u), spread4(h >> 12));
        }
    } else if (mask_vec) {
        for (int o = tid * 16; o < nbytes; o += nthreads * 16) {
            int e0 = o / kNumActions, a0 = o - e0 * kNumActions;
            uint64_t bits = (M[e0] >> a0) | (M[e0 + 1] << (kNumActions - a0));
            uint32_t h = (uint32_t)bits & 0xFFFFu;
            uint4 v = make_uint4(spread4(h & 15u), spread4((h >> 4) & 15u), spread4((h >> 8) & 15u), spread4(h >> 12));
            if (o + 16 <= nbytes) {
                *reinterpret_cast<uint4*>(base + o) = v;
            } else {  // ragged tail of the last tile
                uint32_t w[4] = {v.x, v.y, v.z, v.w};
                for (int b = 0; o + b < nbytes; ++b) base[o + b] = (uint8_t)((w[b >> 2] >> ((b & 3) * 8)) & 1u);
            }
        }
    } else {
        for (int o = tid; o < nbytes; o += nthreads) {
            int e0 = o / kNumActions, a0 = o - e0 * kNumActions;
            base[o] = (uint8_t)((M[e0] >> a0) & 1ull);
        }
    }
}

template <int EPW, int OBS>
__device__ __forceinline__ void emit_tile(const WarpTile<EPW>& t, int lane, int64_t env_base, int n_valid,
                                          void* obs, uint8_t* mask, int mask_vec) {
    if (obs != nullptr)
        for (int e = 0; e < n_valid; ++e) emit_obs_row<OBS>(&t.R[e * kRowStride], lane, obs, env_base + e);
    if (mask != nullptr) emit_mask_run(t.M, lane, 32, mask + env_base * kNumActions, n_valid * kNumActions, mask_vec);
}

// block-cooperative phase 2: the block's warps write the tile's rows interleaved (warp w: rows w, w+W, ...),
// so the addresses a block has in flight stay within a few consecutive rows (scripts/exp_store_paths.cu: a
// pure-write kernel gains 10-15 % when the window of rows in flight per block shrinks from 128 to <= 32)
template <int EPW, int OBS>
__device__ __forceinline__ void emit_block(const WarpTile<EPW>& t, int tid, int nthreads, int64_t env_base, int n_valid,
                                           void* obs, uint8_t* mask, int mask_vec) {
    if (obs != nullptr) {
        const int warp = tid >> 5, lane = tid & 31, nw = nthreads >> 5;
        for (int e = warp; e < n_valid; e += nw) emit_obs_row<OBS>(&t.R[e * kRowStride], lane, obs, env_base + e);
    }
    if (mask != nullptr) emit_mask_run(t.M, tid, nthreads, mask + env_base * kNumActions, n_valid * kNumActions, mask_vec);
}

template <int EPW, class Rows>
__device__ __forceinline__ void stage_env(WarpTile<EPW>& t, int lane, const Env& e, const Rows& rows, uint32_t q,
                                          bool want_obs) {
    if (want_obs) {
        uint32_t R[kObsWords];
        env_observe_words(e, rows, q, R);
#pragma unroll
        for (int w = 0; w < kObsWords; ++w) t.R[lane * kRowStride + w] = R[w];
    }
    t.M[lane] = env_legal_mask(e);
}

__device__ __forceinline__ void write_scalars(const EnvArgs& a, int64_t row, const Env& e, float4 rew, bool accumulate) {
    uint8_t term = (uint8_t)f_terminated(e);
    if (a.rewards) {
        if (accumulate) {
            float4 o = a.rewards[row];
            rew = make_float4(o.x + rew.x, o.y + rew.y, o.z + rew.z, o.w + rew.w);
        }
        a.rewards[row] = rew;
    }
    if (a.terminated) a.terminated[row] = accumulate ? (uint8_t)(a.terminated[row] | term) : term;
    if (a.current_player) a.current_player[row] = (int8_t)f_player_at(e, f_cur_seat(e));
}

#define BRL_TILE_PROLOGUE()                                                          \
    extern __shared__ __align__(16) unsigned char smem_raw[];                        \
    WarpTile<EPW>* tiles = reinterpret_cast<WarpTile<EPW>*>(smem_raw);               \
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;                      \
    const int64_t tile = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;             \
    const int64_t env_base = tile * EPW;                                             \
    if (env_base >= a.n) return;                                                     \
    const int n_valid = (int)((a.n - env_base) < (int64_t)EPW ? (a.n - env_base) : (int64_t)EPW); \
    WarpTile<EPW>& t = tiles[warp];                                                  \
    if (lane < 2) t.M[EPW + lane] = 0ull;                                            \
    const bool active = lane < n_valid;                                              \
    const int64_t i = env_base + lane;

// Block-tile kernels (k_step, k_produce, k_dup_step): a BLOCK owns EPW (<= 32) consecutive envs.  Phase 1 runs
// in the first EPW threads (one env per thread), phase 2 is shared by every warp of the block.
#define BRL_BLOCK_PROLOGUE()                                                         \
    extern __shared__ __align__(16) unsigned char smem_raw[];                        \
    WarpTile<EPW>& t = *reinterpret_cast<WarpTile<EPW>*>(smem_raw);                  \
    const int lane = (int)threadIdx.x;                                               \
    const int64_t env_base = (int64_t)blockIdx.x * EPW;                              \
    const int n_valid = (int)((a.n - env_base) < (int64_t)EPW ? (a.n - env_base) : (int64_t)EPW); \
    if (lane < 2) t.M[EPW + lane] = 0ull;                                            \
    const bool active = lane < n_valid;                                              \
    const int64_t i = env_base + lane;

// ---- one env.step over n envs ---------------------------------------------------------
template <int EPW, int OBS>
__global__ void __launch_bounds__(256) k_step(const EnvArgs a) {
    BRL_BLOCK_PROLOGUE()
    if (lane < EPW) {
        if (active) {
            Env e;
            load_env(a.state_in, a.stride, i, e);
            int32_t act;
            if (a.flags & BRL_F_RANDOM_ACTION) act = random_legal_action(env_legal_mask(e), a.seed, (uint64_t)(a.env_offset + i), a.step);
            else act = a.action[i];
            float4 rew = (a.flags & BRL_F_AUTORESET)
                             ? env_step_autoreset(e, act, a.table, a.n_deals, a.illegal_penalty, a.illegal_bonus)
                             : env_step(e, act, TableRows{a.table}, a.illegal_penalty, a.illegal_bonus);
            const bool acc = (a.flags & BRL_F_ACCUMULATE) != 0;
            if (acc && (a.flags & BRL_F_QUAD_LAST) && a.terminated && (a.terminated[i] || f_terminated(e)))
                e.A |= kTermBit | (f_terminated(e) ? 0u : kCarriedBit);  // src/utils.py:128 state.replace(terminated=OR)
            write_scalars(a, i, e, rew, acc);
            if (a.action_out) a.action_out[i] = act;
            store_env(a.state_out, a.stride, i, e);
            stage_env<EPW>(t, lane, e, TableRows{a.table}, f_cur_seat(e), a.obs != nullptr);
        } else {
            t.M[lane] = 0ull;
        }
    }
    __syncthreads();
    emit_block<EPW, OBS>(t, (int)threadIdx.x, (int)blockDim.x, env_base, n_valid, a.obs, a.mask, a.mask_vec);
}

// caller-supplied action uniform of trajectory row `idx`: u32, or u16 widened to the top half of a u32 (the k-th
// legal action is mulhi(u, #legal), so a 16-bit uniform picks (u16 * #legal) >> 16)
__device__ __forceinline__ uint32_t load_uniform(const EnvArgs& a, int64_t idx) {
    return a.uniform16 ? (uint32_t)reinterpret_cast<const uint16_t*>(a.uniforms)[idx] << 16 : a.uniforms[idx];
}

// warp-specialised rollout: the writer warps fetch the caller's uniforms of steps s0 + 1 .. s0 + kUChunk for the block's envs
// (step r lives in ring slot [(r / kUChunk) & 1][r % kUChunk]; offset d of the burst by warp d % n_writers; every load of a
// warp is issued before the first one is consumed)
constexpr int kUChunk = 32;
__device__ __forceinline__ void load_uniform_burst(const EnvArgs& a, uint32_t (*ring)[kUChunk][32], int s0, int64_t i, bool active,
                                                   int warp, int n_writers, int lane) {
    for (int base = warp; base < kUChunk; base += 8 * n_writers) {
        uint32_t v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int r = s0 + 1 + base + j * n_writers;
            v[j] = (active && base + j * n_writers < kUChunk && r < a.k_steps) ? load_uniform(a, (int64_t)r * a.n + i) : 0u;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int r = s0 + 1 + base + j * n_writers;
            if (base + j * n_writers < kUChunk) ring[(r / kUChunk) & 1][r % kUChunk][lane] = v[j];
        }
    }
}

// compact step result: rewards are s * [+1, +1, -1, -1] by player id with s an integer score in [-7600, 7600]
// (env_device.cuh env_step; no illegal actions on the random-legal path), so 2 * s + terminated is lossless in 16 bits
__device__ __forceinline__ int16_t pack_result16(float rew0, uint32_t term) {
    return (int16_t)(2 * (int)rew0 + (int)(term & 1u));
}

// ---- K auto-reset steps with in-kernel random-legal actions ----------------------------
template <int EPW, int OBS>
__global__ void __launch_bounds__(128) k_rollout(const EnvArgs a) {
    BRL_TILE_PROLOGUE()
    Env e;
    EpisodeCache cache;
    if (active) {
        load_env(a.state_in, a.stride, i, e);
        cache.prime(e, a.table, a.n_deals);
    }
    const size_t obs_row_bytes = OBS == kObsF32 ? kObsDim * 4 : (OBS == kObsU8 ? kObsDim : kObsDim * 2);
    unsigned long long n_term = 0;
    long long rew0 = 0;
    for (int s = 0; s < a.k_steps; ++s) {
        const int64_t row0 = (int64_t)s * a.n;
        if (lane < EPW) {
            if (active) {
                const uint32_t u = a.uniforms ? load_uniform(a, row0 + i)
                                              : action_uniform(a.seed, (uint64_t)(a.env_offset + i), a.step + (uint32_t)s);
                int32_t act = kth_legal_action(env_legal_mask(e), u);
                float4 rew = env_step_autoreset_cached(e, cache, act, a.table, a.n_deals, a.illegal_penalty, a.illegal_bonus);
                n_term += f_terminated(e);
                rew0 += (long long)rew.x;
                write_scalars(a, row0 + i, e, rew, false);
                if (a.result16) a.result16[row0 + i] = pack_result16(rew.x, f_terminated(e));
                if (a.action_out) a.action_out[row0 + i] = act;
                stage_env<EPW>(t, lane, e, cache.cur, f_cur_seat(e), a.obs != nullptr);
            } else {
                t.M[lane] = 0ull;
            }
        }
        __syncwarp();
        emit_tile<EPW, OBS>(t, lane, env_base, n_valid,
                            a.obs ? static_cast<unsigned char*>(a.obs) + (size_t)row0 * obs_row_bytes : nullptr,
                            a.mask ? a.mask + (size_t)row0 * kNumActions : nullptr, a.mask_vec);
        __syncwarp();
    }
    if (active) store_env(a.state_out, a.stride, i, e);
    if (a.stats) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            n_term += __shfl_xor_sync(0xffffffffu, n_term, o);
            rew0 += __shfl_xor_sync(0xffffffffu, rew0, o);
        }
        if (lane == 0) {
            atomicAdd(&a.stats[0], n_term);
            atomicAdd(&a.stats[1], (unsigned long long)rew0);
            atomicAdd(&a.stats[2], (unsigned long long)n_valid * (unsigned long long)a.k_steps);
        }
    }
}

// ---- warp-specialised rollout: 1 env warp + (blockDim/32 - 1) writer warps ---------------
// At 8192 envs every env advances one step per "env-warp step latency" L, so throughput is
// 8192 / L whatever the grouping: the HBM roofline needs L <= ~2.5 us.  The tile-per-warp
// kernel spends L on phase 1 + phase 2 of one warp (ncu: issue-bound on a 36k-instruction
// chain, 6.7 warps/SM).  Here a block owns 32 envs and splits the work by role:
//   env warp (last warp: the issue arbiter favours high warp ids) -- keeps the 32 envs
//     and their deal rows in registers, applies step s and leaves the RAW state words
//     (absolute-seat history, vulnerability nibble, hand bits), the observer seat and the
//     legal mask in one half of a double-buffered shared tile;
//   writer warps -- expand step s-1 from the other half into HBM (nibble-rotate to the
//     observer's seat while expanding, 128-bit coalesced stores), write the per-env
//     scalars, and pre-compute the Philox uniforms of step s+1 for the env warp.
// One __syncthreads per step hands the buffers over.
template <int EPB>
struct WsTile {
    uint32_t R[EPB * kRowStride];  // 15 raw observation words per env (history not yet rotated)
    uint64_t M[EPB + 2];           // legal masks (+2 zero pads)
    float4 rew[EPB];
    uint32_t act[EPB];
    uint8_t q[EPB], term[EPB], cur[EPB];
};

// observation word w for observer seat q from the env warp's RAW words: history nibbles are by absolute
// seat (rotate), the vulnerability nibble (word 0, bits 0-3) and the hand bits (word 13 bits 12+, word 14)
// are already relative to the observer
__device__ __forceinline__ uint32_t obs_word_rot(const uint32_t* R, int w, uint32_t q) {
    const uint32_t v = R[w];
    if (w == 0) return rotr_nibbles(v & ~15u, q) | (v & 15u);
    if (w == 13) return rotr_nibbles(v & 0xFFFu, q) | (v & 0xFFFFF000u);
    if (w == 14) return v;
    return rotr_nibbles(v, q);
}

template <int OBS>
__device__ __forceinline__ void emit_obs_row_rot(const uint32_t* R, uint32_t q, int lane, void* obs, int64_t env) {
    // nibble j of the row: 0 = vulnerability, 1..106 = history (rotate right by q), 107..119 = hand
    if (OBS == kObsF32) {
        float4* row = reinterpret_cast<float4*>(obs) + env * (kObsDim / 4);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int j = lane + 32 * k;
            if (j < kObsDim / 4) {
                uint32_t nib = (R[j >> 3] >> ((j & 7) * 4)) & 15u;
                if (j >= 1 && j <= 106) nib = ((nib | (nib << 4)) >> q) & 15u;
                row[j] = nibble_to_float4(nib);
            }
        }
    } else if (OBS == kObsU8) {
        // u8 row: lane l (< 30) expands 16 bits = half of word l/2; only that word is rotated
        if (lane < kObsDim / 16) {
            uint32_t h = (obs_word_rot(R, lane >> 1, q) >> ((lane & 1) * 16)) & 0xFFFFu;
            reinterpret_cast<uint4*>(obs)[env * (kObsDim / 16) + lane] =
                make_uint4(spread4(h & 15u), spread4((h >> 4) & 15u), spread4((h >> 8) & 15u), spread4(h >> 12));
        }
    } else {
        // bf16 row: 60 uint4 stores of 8 values = one byte of word j/4 each
        uint4* row = reinterpret_cast<uint4*>(obs) + env * (kObsDim / 8);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            int j = lane + 32 * k;
            if (j < kObsDim / 8) {
                uint32_t b = (obs_word_rot(R, j >> 2, q) >> ((j & 3) * 8)) & 0xFFu;
                row[j] = make_uint4(pair_to_bf16x2(b), pair_to_bf16x2(b >> 2), pair_to_bf16x2(b >> 4), pair_to_bf16x2(b >> 6));
            }
        }
    }
}

#ifdef BRL_ROLE_TIMING
__device__ unsigned long long g_role_cycles[8];
// slots 0-5 of g_role_cycles for phase 0 alone (0-5) and the last phase alone (8-13); 6 / 7: the env warp's / warp 0's
// prologue, kernel entry to the end of the first barrier
__device__ unsigned long long g_role_phase_cycles[16];
#define BRL_TP() const long long _tp = clock64()
#define BRL_T0() long long _t0 = clock64(); if (lane == 0 && (is_env_warp || warp == 0)) atomicAdd(&g_role_phase_cycles[is_env_warp ? 6 : 7], (unsigned long long)(_t0 - _tp))
#define BRL_ACC(slot) do { long long _t1 = clock64(); if (lane == 0) { const unsigned long long _d = (unsigned long long)(_t1 - _t0); \
    atomicAdd(&g_role_cycles[slot], _d); \
    if (s == 0) atomicAdd(&g_role_phase_cycles[slot], _d); else if (s == a.k_steps) atomicAdd(&g_role_phase_cycles[8 + (slot)], _d); } \
    _t0 = _t1; } while (0)
#else
#define BRL_TP()
#define BRL_T0()
#define BRL_ACC(slot)
#endif

template <int EPB, int OBS>
__global__ void __launch_bounds__(256) k_rollout_ws(const EnvArgs a) {
    BRL_TP();
    __shared__ WsTile<EPB> tiles[2];
    __shared__ uint32_t uniforms[2][kUChunk][32];  // action uniforms, double-buffered chunks of kUChunk steps
    __shared__ uint4 row_slots[2 * EPB * 3];
    __shared__ unsigned long long row_bars[2 * EPB];
    const RowSlots rs{row_slots, row_bars, EPB};
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_writers = (int)(blockDim.x >> 5) - 1;
    // a.balanced: the grid is a multiple of the SM count and block b owns envs [b*n/G, (b+1)*n/G) (<= EPB of
    // them), so every SM carries the same number of envs even when n / EPB is a small non-multiple of 148
    const int64_t env_base = a.balanced ? ((int64_t)blockIdx.x * a.n) / gridDim.x : (int64_t)blockIdx.x * EPB;
    const int64_t env_end = a.balanced ? ((int64_t)(blockIdx.x + 1) * a.n) / gridDim.x : env_base + EPB;
    const int n_valid = (int)((a.n < env_end ? a.n : env_end) - env_base);
    const bool active = lane < n_valid;
    const int64_t i = env_base + lane;
    const size_t obs_row_bytes = OBS == kObsF32 ? kObsDim * 4 : (OBS == kObsU8 ? kObsDim : kObsDim * 2);
    const bool is_env_warp = warp == n_writers;
    const int mask_mode = a.balanced ? 2 : a.mask_vec;  // mode 2 copes with any alignment of the run
    Env e;
    EpisodePrefetch cache;
    uint64_t mask = 0ull;
    unsigned long long n_term = 0;
    long long rew0 = 0;
    // Launched with programmatic dependent launch (launch_ws_inst): this grid may start while the previous kernel of the
    // stream drains.  Until pdl_wait() only shared memory and pure functions of the arguments are touched: the zero mask
    // pads and, in Philox mode, the uniforms of the first chunk of steps (the writers are idle until the first row).
    pdl_trigger();  // the next launch's blocks take this launch's places as they retire
    const int k_pre = a.uniforms ? 0 : (a.k_steps < kUChunk ? a.k_steps : kUChunk);
    if (is_env_warp) {
        if (lane < 2) { tiles[0].M[EPB + lane] = 0ull; tiles[1].M[EPB + lane] = 0ull; }
    } else {
        for (int r = warp; r < k_pre; r += n_writers)
            uniforms[0][r][lane] = action_uniform(a.seed, (uint64_t)(a.env_offset + i), a.step + (uint32_t)r);
    }
    pdl_wait();  // the previous kernel has completed and its writes (state, deal table, outputs) are visible
    if (is_env_warp) {
        if (active) {
            load_env(a.state_in, a.stride, i, e);
            cache.prime(e, rs, lane, a.table, a.n_deals);
            mask = env_legal_mask(e);
        }
    } else if (warp == 0 && a.uniforms) {
        uniforms[0][0][lane] = active ? load_uniform(a, i) : 0u;
    }
    __syncthreads();
    BRL_T0();
    for (int s = 0; s <= a.k_steps; ++s) {
        if (is_env_warp) {
            if (s < a.k_steps) {
                WsTile<EPB>& t = tiles[s & 1];
                if (active) {
                    int32_t act = kth_legal_action(mask, uniforms[(s / kUChunk) & 1][s % kUChunk][lane]);
                    float4 rew = env_step_autoreset_prefetch(e, cache, rs, lane, act, a.table, a.n_deals, a.illegal_penalty,
                                                             a.illegal_bonus);
                    n_term += f_terminated(e);
                    rew0 += (long long)rew.x;
                    mask = env_legal_mask(e);
                    const uint32_t q = f_cur_seat(e);
                    uint32_t* R = &t.R[lane * kRowStride];
                    if (a.obs) {
                        const uint32_t us = (q & 1u) ? f_vul_ew(e) : f_vul_ns(e), them = (q & 1u) ? f_vul_ns(e) : f_vul_ew(e);
                        const uint64_t hand = cache.cur.hand(e.deal, q);
                        R[0] = e.H[0] | (us ? 2u : 1u) | (them ? 8u : 4u);
#pragma unroll
                        for (int w = 1; w < 13; ++w) R[w] = e.H[w];
                        R[13] = e.H[13] | (uint32_t)(hand << 12);
                        R[14] = (uint32_t)(hand >> 20);
                    }
                    t.M[lane] = mask;
                    t.rew[lane] = rew;
                    t.act[lane] = (uint32_t)act;
                    t.q[lane] = (uint8_t)q;
                    t.term[lane] = (uint8_t)f_terminated(e);
                    t.cur[lane] = (uint8_t)f_player_at(e, q);
                } else if (lane < EPB) {
                    t.M[lane] = 0ull;
                }
            }
        } else {
            if (s > 0) {
                const WsTile<EPB>& t = tiles[(s - 1) & 1];
                const int64_t row0 = (int64_t)(s - 1) * a.n;
                if (a.obs) {
                    unsigned char* obs = static_cast<unsigned char*>(a.obs) + (size_t)row0 * obs_row_bytes;
                    // two rows in flight per warp: the second row's shared loads and expansion fill the first row's store / dependency
                    // stalls (measured 91.6 -> 89.4 us per launch at the bench shape; four rows: 94.2, scripts/exp_lib_variants.py)
#pragma unroll 2
                    for (int r = warp; r < n_valid; r += n_writers)
                        emit_obs_row_rot<OBS>(&t.R[r * kRowStride], t.q[r], lane, obs, env_base + r);
                }
                if (a.mask)
                    emit_mask_run(t.M, (int)threadIdx.x, n_writers * 32, a.mask + (size_t)(row0 + env_base) * kNumActions,
                                  n_valid * kNumActions, mask_mode);
                if (warp == n_writers - 1 && active) {  // per-env scalars, coalesced over the tile
                    const int64_t row = row0 + i;
                    if (a.rewards) a.rewards[row] = t.rew[lane];
                    if (a.terminated) a.terminated[row] = t.term[lane];
                    if (a.result16) a.result16[row] = pack_result16(t.rew[lane].x, t.term[lane]);
                    if (a.current_player) a.current_player[row] = (int8_t)t.cur[lane];
                    if (a.action_out) a.action_out[row] = (int32_t)t.act[lane];
                }
            }
            if (s + 1 < a.k_steps) {
                if (a.uniforms) {
                    // Caller-supplied uniforms are read in bursts of kUChunk steps, every warp's loads in flight at once: a
                    // 128-byte read per block per step, trickling into DRAM between the trajectory's writes, cost 6-13 % of
                    // the whole kernel (read / write turnarounds; the pool is evicted from L2 by the 519 MB a launch
                    // writes), scripts/exp_e2e_gap.py.  The burst for steps s+1 .. s+32 is issued at s = 0, 32, ...: at s = 0
                    // the writers have nothing to store yet, so it hides under the env warp's first step.
                    if (s % kUChunk == 0) load_uniform_burst(a, uniforms, s, i, active, warp, n_writers, lane);
                } else if (warp == 0 && s + 1 >= kUChunk) {  // the first chunk was drawn before pdl_wait()
                    uniforms[((s + 1) / kUChunk) & 1][(s + 1) % kUChunk][lane] =
                        action_uniform(a.seed, (uint64_t)(a.env_offset + i), a.step + (uint32_t)(s + 1));
                }
            }
        }
        BRL_ACC(is_env_warp ? 0 : (warp == 0 ? 2 : 4));
        __syncthreads();
        BRL_ACC(is_env_warp ? 1 : (warp == 0 ? 3 : 5));
    }
    if (is_env_warp) {
        if (active) store_env(a.state_out, a.stride, i, e);
        asm volatile("cp.async.wait_all;" ::: "memory");  // the last prefetch must land before the block's smem is released
        if (a.stats) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                n_term += __shfl_xor_sync(0xffffffffu, n_term, o);
                rew0 += __shfl_xor_sync(0xffffffffu, rew0, o);
            }
            if (lane == 0) {
                atomicAdd(&a.stats[0], n_term);
                atomicAdd(&a.stats[1], (unsigned long long)rew0);
                atomicAdd(&a.stats[2], (unsigned long long)n_valid * (unsigned long long)a.k_steps);
            }
        }
    }
}

// ---- init / reset_fields / duplicate_init / observe / legal_mask -----------------------
enum ProduceMode { kModeInit = 0, kModeReset = 1, kModeDupInit = 2, kModeObserve = 3 };

template <int EPW, int OBS>
__global__ void __launch_bounds__(256) k_produce(const EnvArgs a) {
    BRL_BLOCK_PROLOGUE()
    if (lane < EPW) {
        if (active) {
            Env e;
            uint32_t q;
            if (a.mode == kModeInit) {
                env_init(e, a.keys[i], a.n_deals);
            } else if (a.mode == kModeReset) {
                const int8_t* p = a.in_players + 4 * i;
                uint32_t seating8 = (uint32_t)(p[0] & 3) | ((uint32_t)(p[1] & 3) << 2) | ((uint32_t)(p[2] & 3) << 4) |
                                    ((uint32_t)(p[3] & 3) << 6);
                env_reset(e, (uint32_t)a.in_deal[i], (uint32_t)a.in_dealer[i] & 3u, a.in_vul_ns[i] ? 1u : 0u,
                          a.in_vul_ew[i] ? 1u : 0u, seating8, a.in_rng_key ? a.in_rng_key[i] : 0ull);
            } else {
                load_env(a.state_in, a.stride, i, e);
                if (a.mode == kModeDupInit) env_duplicate_init(e);
            }
            q = f_cur_seat(e);
            if (a.mode == kModeObserve && a.in_player_id) {  // _observe(state, player): seat of that player id
                uint32_t pid = (uint32_t)a.in_player_id[i] & 3u;
#pragma unroll
                for (uint32_t s = 0; s < 4; ++s)
                    if (f_player_at(e, s) == pid) q = s;
            }
            if (a.mode <= kModeDupInit) {
                store_env(a.state_out, a.stride, i, e);
                write_scalars(a, i, e, make_float4(0.f, 0.f, 0.f, 0.f), false);
            }
            stage_env<EPW>(t, lane, e, TableRows{a.table}, q, a.obs != nullptr);
        } else {
            t.M[lane] = 0ull;
        }
    }
    __syncthreads();
    emit_block<EPW, OBS>(t, (int)threadIdx.x, (int)blockDim.x, env_base, n_valid, a.obs, a.mask, a.mask_vec);
}

// ---- legal_action_mask alone -------------------------------------------------------------
// The mask is a function of state word A alone (one 16-byte plane read per env; 38 bytes out).  A block owns 256
// consecutive envs: every thread turns one A into 38 mask bits in shared memory, then the block writes its
// 256 * 38 = 9728 output bytes as 608 fully coalesced 128-bit stores (each one assembled from at most two envs).
constexpr int kMaskEnvsPerBlock = 256;

__global__ void __launch_bounds__(kMaskEnvsPerBlock) k_legal_mask(const uint4* __restrict__ state, int64_t stride,
                                                                   uint8_t* __restrict__ mask, int64_t n, int vec) {
    __shared__ uint64_t M[kMaskEnvsPerBlock + 2];
    const int tid = (int)threadIdx.x;
    const int64_t env_base = (int64_t)blockIdx.x * kMaskEnvsPerBlock;
    const int n_valid = (int)((n - env_base) < (int64_t)kMaskEnvsPerBlock ? (n - env_base) : (int64_t)kMaskEnvsPerBlock);
    uint64_t m = 0ull;
    if (tid < n_valid) {
        Env e = {};
        e.A = state[3 * stride + env_base + tid].z;
        m = env_legal_mask(e);
    }
    M[tid] = m;
    if (tid < 2) M[kMaskEnvsPerBlock + tid] = 0ull;
    __syncthreads();
    emit_mask_run(M, tid, kMaskEnvsPerBlock, mask + env_base * kNumActions, n_valid * kNumActions, vec);
}

// ---- duplicate_step -- src/duplicate.py:147-192 ----------------------------------------
template <int EPW, int OBS>
__global__ void __launch_bounds__(256) k_dup_step(const EnvArgs a) {
    BRL_BLOCK_PROLOGUE()
    if (lane < EPW) {
        if (active) {
            Env e;
            load_env(a.state_in, a.stride, i, e);
            float4 rew = env_step(e, a.action[i], TableRows{a.table}, a.illegal_penalty, a.illegal_bonus);  // :149
            const bool term = f_terminated(e) != 0;
            const bool a_term = a.ta.terminated[i] != 0, b_term = a.tb.terminated[i] != 0;
            const bool a_just = !a_term && term;           // :152
            const bool b_just = a_term && term && !b_term;  // :158
            // snapshot of the stepped state (:165-188)
            const uint32_t lb1 = f_lb1(e);
            const int32_t s_last_bid = (int32_t)lb1 - 1;
            const int32_t s_last_bidder = lb1 ? (int32_t)f_player_at(e, f_bidder_seat(e)) : -1;
            const uint8_t s_x = (uint8_t)f_x(e), s_xx = (uint8_t)f_xx(e);
            float4 out_rew = make_float4(0.f, 0.f, 0.f, 0.f);
            if (b_just) {
                float s = imp_of_difference(a.ta.rewards[i].x + rew.x);  // :159-161, _imp_reward :15-70
                out_rew = make_float4(s, s, -s, -s);
            } else if (a_just) {
                env_duplicate_init(e);  // :151-155
            }
            if (a_just || b_just) {
                const TableInfo& ti = b_just ? a.tb : a.ta;
                ti.terminated[i] = 1;
                ti.rewards[i] = rew;
                ti.last_bid[i] = s_last_bid;
                ti.last_bidder[i] = s_last_bidder;
                ti.call_x[i] = s_x;
                ti.call_xx[i] = s_xx;
            }
            write_scalars(a, i, e, out_rew, false);
            store_env(a.state_out, a.stride, i, e);
            stage_env<EPW>(t, lane, e, TableRows{a.table}, f_cur_seat(e), a.obs != nullptr);
        } else {
            t.M[lane] = 0ull;
        }
    }
    __syncthreads();
    emit_block<EPW, OBS>(t, (int)threadIdx.x, (int)blockDim.x, env_base, n_valid, a.obs, a.mask, a.mask_vec);
}

// ---- private field export ----------------------------------------------------------------
struct FieldArgs {
    const uint4* state;
    int32_t* deal;
    int32_t* dealer;
    int8_t* shuffled;
    uint8_t* vul;
    int32_t* last_bid;
    int32_t* last_bidder;
    uint8_t* call_x;
    uint8_t* call_xx;
    int32_t* pass_num;
    int32_t* step_count;
    uint64_t* rng_key;
    int64_t n, stride;
};

__global__ void __launch_bounds__(256) k_state_fields(const FieldArgs a) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    Env e;
    load_env(a.state, a.stride, i, e);
    if (a.deal) a.deal[i] = (int32_t)e.deal;
    if (a.dealer) a.dealer[i] = (int32_t)f_dealer(e);
    if (a.shuffled) {
        char4 p = make_char4((char)f_player_at(e, 0), (char)f_player_at(e, 1), (char)f_player_at(e, 2), (char)f_player_at(e, 3));
        reinterpret_cast<char4*>(a.shuffled)[i] = p;
    }
    if (a.vul) reinterpret_cast<uchar2*>(a.vul)[i] = make_uchar2((unsigned char)f_vul_ns(e), (unsigned char)f_vul_ew(e));
    uint32_t lb1 = f_lb1(e);
    if (a.last_bid) a.last_bid[i] = (int32_t)lb1 - 1;
    if (a.last_bidder) a.last_bidder[i] = lb1 ? (int32_t)f_player_at(e, f_bidder_seat(e)) : -1;
    if (a.call_x) a.call_x[i] = (uint8_t)f_x(e);
    if (a.call_xx) a.call_xx[i] = (uint8_t)f_xx(e);
    if (a.pass_num) a.pass_num[i] = (int32_t)f_pass_num(e);
    if (a.step_count) a.step_count[i] = (int32_t)f_step_count(e);
    if (a.rng_key) a.rng_key[i] = (uint64_t)e.key_lo | ((uint64_t)e.key_hi << 32);
}

__global__ void __launch_bounds__(256) k_make_keys(uint64_t* keys, int64_t n, uint64_t seed, int64_t env_offset) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = make_key(seed, (uint64_t)(env_offset + i));
}

// ---- launch helpers ---------------------------------------------------------------------------
struct Tiling {
    int epw, wpb;
};

static Tiling choose_tiling(int64_t n, int32_t flags) {
    // flags bits 16-17: EPW override (1->8, 2->16, 3->32); bits 18-19: warps per block (1->1, 2->2, 3->4; with
    // bit 26 also set: 8)
    static const int epw_of[4] = {0, 8, 16, 32};
    static const int wpb_of[4] = {0, 1, 2, 4};
    int epw = epw_of[(flags >> 16) & 3], wpb = wpb_of[(flags >> 18) & 3];
    if (wpb && (flags & (1 << 26))) wpb = 8;
    if (epw == 0) epw = n >= 262144 ? 32 : (n >= 65536 ? 16 : 8);  // >= ~8 warps per SM at every size
    if (wpb == 0) wpb = n >= 65536 ? 4 : 2;
    return {epw, wpb};
}

// block-tile kernels: envs per block (8/16/32) and warps per block (1..8) sharing its phase 2
static Tiling choose_block_tiling(int64_t n, int32_t flags) {
    Tiling t = choose_tiling(n, flags);
    // measured at 1,048,576 envs (scripts/exp_tiling.py): the fewer rows a block has in flight, the closer the stores
    // get to the pure-write ceiling, until phase 1 (EPW of the block's threads busy) starves it; 480-byte u8 rows
    // need twice the envs per block for the same bytes in flight
    if (((flags >> 16) & 3) == 0) t.epw = ((flags & BRL_F_OBS_U8) && n >= 262144) ? 32 : 16;
    if (((flags >> 18) & 3) == 0) t.wpb = 4;
    return t;
}

#define BRL_DEFINE_LAUNCHER(NAME, KERNEL)                                                                    \
    template <int EPW, int OBS>                                                                              \
    static void NAME##_inst(const EnvArgs& a, int wpb, cudaStream_t s) {                                     \
        int64_t tiles = (a.n + EPW - 1) / EPW;                                                               \
        unsigned grid = (unsigned)((tiles + wpb - 1) / wpb);                                                 \
        KERNEL<EPW, OBS><<<grid, wpb * 32, wpb * sizeof(WarpTile<EPW>), s>>>(a);                             \
    }                                                                                                        \
    template <int OBS>                                                                                       \
    static void NAME##_epw(const EnvArgs& a, Tiling t, cudaStream_t s) {                                     \
        if (t.epw == 8) NAME##_inst<8, OBS>(a, t.wpb, s);                                                    \
        else if (t.epw == 16) NAME##_inst<16, OBS>(a, t.wpb, s);                                             \
        else NAME##_inst<32, OBS>(a, t.wpb, s);                                                              \
    }                                                                                                        \
    static void NAME(const EnvArgs& a, cudaStream_t s) {                                                     \
        if (a.n == 0) return;                                                                                \
        Tiling t = choose_tiling(a.n, a.flags);                                                              \
        if (a.flags & BRL_F_OBS_U8) NAME##_epw<kObsU8>(a, t, s);                                             \
        else if (a.flags & BRL_F_OBS_BF16) NAME##_epw<kObsBF16>(a, t, s);                                    \
        else NAME##_epw<kObsF32>(a, t, s);                                                                   \
    }

BRL_DEFINE_LAUNCHER(launch_rollout, k_rollout)

#define BRL_DEFINE_BLOCK_LAUNCHER(NAME, KERNEL)                                                              \
    template <int EPW, int OBS>                                                                              \
    static void NAME##_inst(const EnvArgs& a, int wpb, cudaStream_t s) {                                     \
        unsigned grid = (unsigned)((a.n + EPW - 1) / EPW);                                                   \
        KERNEL<EPW, OBS><<<grid, wpb * 32, sizeof(WarpTile<EPW>), s>>>(a);                                   \
    }                                                                                                        \
    template <int OBS>                                                                                       \
    static void NAME##_epw(const EnvArgs& a, Tiling t, cudaStream_t s) {                                     \
        if (t.epw == 8) NAME##_inst<8, OBS>(a, t.wpb, s);                                                    \
        else if (t.epw == 16) NAME##_inst<16, OBS>(a, t.wpb, s);                                             \
        else NAME##_inst<32, OBS>(a, t.wpb, s);                                                              \
    }                                                                                                        \
    static void NAME(const EnvArgs& a, cudaStream_t s) {                                                     \
        if (a.n == 0) return;                                                                                \
        Tiling t = choose_block_tiling(a.n, a.flags);                                                        \
        if (a.flags & BRL_F_OBS_U8) NAME##_epw<kObsU8>(a, t, s);                                             \
        else if (a.flags & BRL_F_OBS_BF16) NAME##_epw<kObsBF16>(a, t, s);                                    \
        else NAME##_epw<kObsF32>(a, t, s);                                                                   \
    }

BRL_DEFINE_BLOCK_LAUNCHER(launch_step, k_step)
BRL_DEFINE_BLOCK_LAUNCHER(launch_produce, k_produce)
BRL_DEFINE_BLOCK_LAUNCHER(launch_dup_step, k_dup_step)

// flags bit 20: force the tile-per-warp rollout kernel; bits 16-17: envs per block of the
// warp-specialised kernel (as EPW); bits 21-23: its writer warps (0 = auto, else the count).
template <int EPB, int OBS>
static void launch_ws_inst(const EnvArgs& a, int writers, cudaStream_t s) {
    unsigned grid = (unsigned)((a.n + EPB - 1) / EPB);
    if (a.balanced) grid = ((grid + 147u) / 148u) * 148u;  // 148 SMs: same number of blocks on every SM
    // every launch waits (pdl_wait) for the complete previous kernel of the stream, so an event or kernel after a
    // chain of rollouts still sees all of them finished
    launch_pdl(k_rollout_ws<EPB, OBS>, dim3(grid), dim3(32 * (1 + writers)), 0, s, a);
}
template <int OBS>
static void launch_ws_obs(const EnvArgs& a, int epb, int writers, cudaStream_t s) {
    if (epb == 8) launch_ws_inst<8, OBS>(a, writers, s);
    else if (epb == 16) launch_ws_inst<16, OBS>(a, writers, s);
    else launch_ws_inst<32, OBS>(a, writers, s);
}
static void launch_rollout_ws(const EnvArgs& a_in, cudaStream_t s) {
    if (a_in.n == 0) return;
    EnvArgs a = a_in;
    // flags bit 24: force the balanced split on, bit 25: force it off; auto = on when the plain grid would
    // leave some SMs with >= 10 % more blocks than others (few blocks per SM)
    {
        const int64_t blocks = (a.n + 31) / 32;
        const int64_t per_sm_hi = (blocks + 147) / 148;
        const bool uneven = blocks % 148 != 0 && per_sm_hi <= 8 && blocks >= 148;
        a.balanced = (a.flags & (1 << 24)) ? 1 : ((a.flags & (1 << 25)) ? 0 : (uneven ? 1 : 0));
    }
    static const int epb_of[4] = {0, 8, 16, 32};
    int epb = epb_of[(a.flags >> 16) & 3];
    if (epb == 0) epb = a.n < 8192 ? 16 : 32;  // measured (scripts/exp_rollout_shapes.py)
    int writers = (a.flags >> 21) & 7;
    // measured: scripts/exp_ab.py, and for the balanced grid scripts/exp_compressible.py: into compressible trajectories seven
    // writers beat four (82.4 against 88.6 us per launch at 8192 envs x 32 steps, B200 at 1000 W); into plain memory seven
    // would lose (98.5 against 89.0 us), as the extra issue rate there only meets the DRAM write-back that compression shrinks
    if (writers == 0) writers = epb == 8 ? 1 : (epb == 16 ? 2 : (a.balanced ? 7 : 3));
    if (a.flags & BRL_F_OBS_U8) launch_ws_obs<kObsU8>(a, epb, writers, s);
    else if (a.flags & BRL_F_OBS_BF16) launch_ws_obs<kObsBF16>(a, epb, writers, s);
    else launch_ws_obs<kObsF32>(a, epb, writers, s);
}

static void fill_common(EnvArgs& a, const BrlParams* p) {
    a.n = p->n_envs;
    a.stride = p->state_stride > 0 ? p->state_stride : p->n_envs;
    a.env_offset = p->env_offset;
    a.seed = p->seed;
    a.n_deals = (uint32_t)p->n_deals;
    a.step = p->step;
    a.flags = p->flags;
    a.k_steps = p->k_steps;
    a.illegal_penalty = p->illegal_penalty;
    a.illegal_bonus = p->illegal_bonus;
}

static int mask_vec_ok(const void* mask, int64_t n, int rows) {
    if (mask == nullptr) return 0;
    if (reinterpret_cast<uintptr_t>(mask) & 15u) return 0;
    return rows <= 1 || ((n * kNumActions) % 16 == 0);
}

static void set_outputs(EnvArgs& a, void** b, int first, int rows) {
    a.obs = b[first];
    a.mask = static_cast<uint8_t*>(b[first + 1]);
    a.rewards = static_cast<float4*>(b[first + 2]);
    a.terminated = static_cast<uint8_t*>(b[first + 3]);
    a.current_player = static_cast<int8_t*>(b[first + 4]);
    a.mask_vec = mask_vec_ok(a.mask, a.n, rows);
}

static int32_t check_outputs(const EnvArgs& a, const char* fn) {
    if (a.obs && (reinterpret_cast<uintptr_t>(a.obs) & 15u)) return fail(BRL_E_BUFFER, "%s: obs is not 16-byte aligned", fn);
    if (a.rewards && (reinterpret_cast<uintptr_t>(a.rewards) & 15u)) return fail(BRL_E_BUFFER, "%s: rewards is not 16-byte aligned", fn);
    return BRL_OK;
}

static TableInfo table_info(void** b, int first) {
    TableInfo t;
    t.terminated = static_cast<uint8_t*>(b[first]);
    t.rewards = static_cast<float4*>(b[first + 1]);
    t.last_bid = static_cast<int32_t*>(b[first + 2]);
    t.last_bidder = static_cast<int32_t*>(b[first + 3]);
    t.call_x = static_cast<uint8_t*>(b[first + 4]);
    t.call_xx = static_cast<uint8_t*>(b[first + 5]);
    return t;
}

}  // namespace brl

using namespace brl;

extern "C" {

int32_t brl_make_keys(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "keys");
    k_make_keys<<<(unsigned)((p->n_envs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        static_cast<uint64_t*>(b[0]), p->n_envs, p->seed, p->env_offset);
    return check_launch("brl_make_keys");
}

int32_t brl_init(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "keys");
    BRL_REQUIRE(b[1], "deal_table");
    BRL_REQUIRE(b[2], "state_out");
    if (p->n_deals <= 0) return fail(BRL_E_OPAQUE, "brl_init: n_deals must be > 0");
    EnvArgs a = {};
    fill_common(a, p);
    a.mode = kModeInit;
    a.keys = static_cast<const uint64_t*>(b[0]);
    a.table = static_cast<const uint8_t*>(b[1]);
    a.state_out = static_cast<uint4*>(b[2]);
    set_outputs(a, b, 3, 1);
    if ((rc = check_outputs(a, "brl_init")) != BRL_OK) return rc;
    launch_produce(a, (cudaStream_t)stream);
    return check_launch("brl_init");
}

int32_t brl_reset_fields(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    static const char* names[] = {"deal", "dealer", "vul_ns", "vul_ew", "shuffled_players"};
    for (int k = 0; k < 5; ++k)
        if (b[k] == nullptr) return fail(BRL_E_BUFFER, "brl_reset_fields: buffer '%s' is NULL", names[k]);
    BRL_REQUIRE(b[6], "deal_table");
    BRL_REQUIRE(b[7], "state_out");
    EnvArgs a = {};
    fill_common(a, p);
    a.mode = kModeReset;
    a.in_deal = static_cast<const int32_t*>(b[0]);
    a.in_dealer = static_cast<const int32_t*>(b[1]);
    a.in_vul_ns = static_cast<const uint8_t*>(b[2]);
    a.in_vul_ew = static_cast<const uint8_t*>(b[3]);
    a.in_players = static_cast<const int8_t*>(b[4]);
    a.in_rng_key = static_cast<const uint64_t*>(b[5]);
    a.table = static_cast<const uint8_t*>(b[6]);
    a.state_out = static_cast<uint4*>(b[7]);
    set_outputs(a, b, 8, 1);
    if ((rc = check_outputs(a, "brl_reset_fields")) != BRL_OK) return rc;
    launch_produce(a, (cudaStream_t)stream);
    return check_launch("brl_reset_fields");
}

int32_t brl_step(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "state_in");
    if (!(p->flags & BRL_F_RANDOM_ACTION) && b[1] == nullptr) return fail(BRL_E_BUFFER, "brl_step: buffer 'action' is NULL");
    BRL_REQUIRE(b[2], "deal_table");
    BRL_REQUIRE(b[3], "state_out");
    if ((p->flags & BRL_F_AUTORESET) && p->n_deals <= 0) return fail(BRL_E_OPAQUE, "brl_step: n_deals must be > 0 with BRL_F_AUTORESET");
    EnvArgs a = {};
    fill_common(a, p);
    a.state_in = static_cast<const uint4*>(b[0]);
    a.action = static_cast<const int32_t*>(b[1]);
    a.table = static_cast<const uint8_t*>(b[2]);
    a.state_out = static_cast<uint4*>(b[3]);
    set_outputs(a, b, 4, 1);
    a.action_out = static_cast<int32_t*>(b[9]);
    if ((rc = check_outputs(a, "brl_step")) != BRL_OK) return rc;
    launch_step(a, (cudaStream_t)stream);
    return check_launch("brl_step");
}

int32_t brl_duplicate_step(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "state_in");
    if (b[1] == nullptr) return fail(BRL_E_BUFFER, "brl_duplicate_step: buffer 'action' is NULL");
    BRL_REQUIRE(b[2], "deal_table");
    for (int k = 3; k < 15; ++k)
        if (b[k] == nullptr) return fail(BRL_E_BUFFER, "brl_duplicate_step: table-info buffer %d is NULL", k);
    BRL_REQUIRE(b[4], "table_a.rewards");
    BRL_REQUIRE(b[10], "table_b.rewards");
    BRL_REQUIRE(b[15], "state_out");
    EnvArgs a = {};
    fill_common(a, p);
    a.state_in = static_cast<const uint4*>(b[0]);
    a.action = static_cast<const int32_t*>(b[1]);
    a.table = static_cast<const uint8_t*>(b[2]);
    a.ta = table_info(b, 3);
    a.tb = table_info(b, 9);
    a.state_out = static_cast<uint4*>(b[15]);
    set_outputs(a, b, 16, 1);
    if ((rc = check_outputs(a, "brl_duplicate_step")) != BRL_OK) return rc;
    launch_dup_step(a, (cudaStream_t)stream);
    return check_launch("brl_duplicate_step");
}

int32_t brl_duplicate_init(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "state_in");
    BRL_REQUIRE(b[1], "deal_table");
    BRL_REQUIRE(b[2], "state_out");
    EnvArgs a = {};
    fill_common(a, p);
    a.mode = kModeDupInit;
    a.state_in = static_cast<const uint4*>(b[0]);
    a.table = static_cast<const uint8_t*>(b[1]);
    a.state_out = static_cast<uint4*>(b[2]);
    set_outputs(a, b, 3, 1);
    if ((rc = check_outputs(a, "brl_duplicate_init")) != BRL_OK) return rc;
    launch_produce(a, (cudaStream_t)stream);
    return check_launch("brl_duplicate_init");
}

int32_t brl_observe(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "state");
    BRL_REQUIRE(b[2], "deal_table");
    BRL_REQUIRE(b[3], "obs");
    EnvArgs a = {};
    fill_common(a, p);
    a.mode = kModeObserve;
    a.state_in = static_cast<const uint4*>(b[0]);
    a.in_player_id = static_cast<const int8_t*>(b[1]);
    a.table = static_cast<const uint8_t*>(b[2]);
    a.obs = b[3];
    launch_produce(a, (cudaStream_t)stream);
    return check_launch("brl_observe");
}

int32_t brl_legal_mask(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "state");
    if (b[1] == nullptr) return fail(BRL_E_BUFFER, "brl_legal_mask: buffer 'mask' is NULL");
    EnvArgs a = {};
    fill_common(a, p);
    a.state_in = static_cast<const uint4*>(b[0]);
    a.mask = static_cast<uint8_t*>(b[1]);
    // 256 * 38 bytes per block is a multiple of 16, so every block's run starts 16-byte aligned when the buffer is
    k_legal_mask<<<(unsigned)((a.n + kMaskEnvsPerBlock - 1) / kMaskEnvsPerBlock), kMaskEnvsPerBlock, 0, (cudaStream_t)stream>>>(
        a.state_in, a.stride, a.mask, a.n, mask_vec_ok(a.mask, a.n, 1));
    return check_launch("brl_legal_mask");
}

int32_t brl_rollout_random(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "state");
    BRL_REQUIRE(b[1], "deal_table");
    if (p->k_steps <= 0) return fail(BRL_E_OPAQUE, "brl_rollout_random: k_steps must be > 0");
    if (p->n_deals <= 0) return fail(BRL_E_OPAQUE, "brl_rollout_random: n_deals must be > 0");
    EnvArgs a = {};
    fill_common(a, p);
    a.state_in = static_cast<const uint4*>(b[0]);
    a.state_out = static_cast<uint4*>(b[0]);
    a.table = static_cast<const uint8_t*>(b[1]);
    set_outputs(a, b, 2, p->k_steps);
    a.action_out = static_cast<int32_t*>(b[7]);
    a.stats = static_cast<unsigned long long*>(b[8]);
    a.uniforms = static_cast<const uint32_t*>(b[9]);
    a.uniform16 = (p->flags & BRL_F_UNIFORM_U16) ? 1 : 0;
    if (a.uniforms && (reinterpret_cast<uintptr_t>(a.uniforms) & (a.uniform16 ? 1u : 3u)))
        return fail(BRL_E_BUFFER, "brl_rollout_random: uniforms is misaligned for its element type");
    if (p->flags & BRL_F_RESULT_I16) {
        a.result16 = static_cast<int16_t*>(b[10]);
        if (a.result16 == nullptr || (reinterpret_cast<uintptr_t>(a.result16) & 1u))
            return fail(BRL_E_BUFFER, "brl_rollout_random: BRL_F_RESULT_I16 needs an i16-aligned buffer [10]");
    }
    if ((rc = check_outputs(a, "brl_rollout_random")) != BRL_OK) return rc;
    if (p->flags & (1 << 20)) launch_rollout(a, (cudaStream_t)stream);
    else launch_rollout_ws(a, (cudaStream_t)stream);
    return check_launch("brl_rollout_random");
}

int32_t brl_state_fields(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "state");
    FieldArgs a;
    a.state = static_cast<const uint4*>(b[0]);
    a.deal = static_cast<int32_t*>(b[1]);
    a.dealer = static_cast<int32_t*>(b[2]);
    a.shuffled = static_cast<int8_t*>(b[3]);
    a.vul = static_cast<uint8_t*>(b[4]);
    a.last_bid = static_cast<int32_t*>(b[5]);
    a.last_bidder = static_cast<int32_t*>(b[6]);
    a.call_x = static_cast<uint8_t*>(b[7]);
    a.call_xx = static_cast<uint8_t*>(b[8]);
    a.pass_num = static_cast<int32_t*>(b[9]);
    a.step_count = static_cast<int32_t*>(b[10]);
    a.rng_key = static_cast<uint64_t*>(b[11]);
    a.n = p->n_envs;
    a.stride = p->state_stride > 0 ? p->state_stride : p->n_envs;
    k_state_fields<<<(unsigned)((a.n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
    return check_launch("brl_state_fields");
}

#ifdef BRL_ROLE_TIMING
// debug build only: cycles spent {env work, env barrier, writer0 work, writer0 barrier, other writers work, barrier}
int32_t brl_debug_role_cycles(unsigned long long* out8, int reset) {
    cudaMemcpyFromSymbol(out8, g_role_cycles, sizeof(g_role_cycles));
    if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(g_role_cycles, z, sizeof(z)); }
    return 0;
}
// the same split by phase: {phase 0: slots 0-5, prologue: 6-7, last phase: 8-13} (g_role_phase_cycles)
int32_t brl_debug_role_phase_cycles(unsigned long long* out16, int reset) {
    cudaMemcpyFromSymbol(out16, g_role_phase_cycles, sizeof(g_role_phase_cycles));
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(g_role_phase_cycles, z, sizeof(z)); }
    return 0;
}
#endif

}  // extern "C"

// ---- brl_sl_examples: supervised-learning examples (make_dataset, sl.py:100-117) ---------------------------------------
// A tile kernel like k_produce: phase 1 replays one stored auction prefix per lane with env_reset / env_step, phase 2 is
// the block's emit_block.  BRL_F_SL_CHECK replays every whole auction once and writes a status byte per trajectory.
namespace brl {

// The dataset's deals: OpenSpiel's bridge(use_double_dummy_result=false) (sl.py:44) has dealer North, nobody vulnerable,
// and players identical to seats.
constexpr uint32_t kSlSeating = 0u | (1u << 2) | (2u << 4) | (3u << 6);
constexpr uint32_t kTagSl = 0x534C3030u;  // "SL00": Philox stream of the call positions

struct SlArgs {
    const uint8_t* table;      // one 48-byte deal row per trajectory
    const uint8_t* calls;      // call actions 0..37, trajectory t at [offsets[t], offsets[t + 1])
    const int64_t* offsets;    // [n_traj + 1]
    const int32_t* traj;       // [B]
    const int32_t* position;   // [B] or NULL: uniform in [0, n_calls) from Philox(seed; example, step)
    void* obs;
    uint8_t* mask;
    int32_t* label;
    int32_t* position_out;     // optional
    uint8_t* status;           // check mode: [n_traj]
    int64_t n, env_offset, n_traj;
    uint64_t seed;
    uint32_t step;
    int mask_vec;
};

__device__ __forceinline__ void sl_reset(Env& e, uint32_t t) { env_reset(e, t, 0u, 0u, 0u, kSlSeating, 0ull); }

// sl.py:106: np.random.randint(52, len(trajectory)) -- a call position uniform in [0, n_calls)
__device__ __forceinline__ int32_t sl_position(uint64_t seed, uint64_t example, uint32_t step, int64_t n_calls) {
    const uint32_t r = philox4x32(make_uint4((uint32_t)example, (uint32_t)(example >> 32), kTagSl, step),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32))).x;
    return (int32_t)__umulhi(r, (uint32_t)n_calls);
}

template <int EPW, int OBS>
__global__ void __launch_bounds__(256) k_sl_examples(const SlArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WarpTile<EPW>& t = *reinterpret_cast<WarpTile<EPW>*>(smem_raw);
    const int lane = (int)threadIdx.x;
    const int64_t env_base = (int64_t)blockIdx.x * EPW;
    const int n_valid = (int)((a.n - env_base) < (int64_t)EPW ? (a.n - env_base) : (int64_t)EPW);
    if (lane < 2) t.M[EPW + lane] = 0ull;
    const int64_t i = env_base + lane;
    // phase 1: one example per lane
    if (lane < EPW) {
        if (lane < n_valid) {
            const uint32_t tr = (uint32_t)a.traj[i];
            const int64_t off = a.offsets[tr], n_calls = a.offsets[tr + 1] - off;
            int32_t pos = a.position ? a.position[i] : sl_position(a.seed, (uint64_t)(a.env_offset + i), a.step, n_calls);
            const bool in_range = pos >= 0 && pos < n_calls;
            if (!in_range) pos = pos < 0 ? 0 : (int32_t)n_calls;  // label -1 marks a position outside the auction
            Env e;
            sl_reset(e, tr);
            for (int32_t k = 0; k < pos; ++k) env_step(e, (int32_t)a.calls[off + k], TableRows{a.table}, -1.0f, 1.0f);
            a.label[i] = in_range ? (int32_t)a.calls[off + pos] : -1;
            if (a.position_out) a.position_out[i] = in_range ? pos : -1;
            stage_env<EPW>(t, lane, e, TableRows{a.table}, f_cur_seat(e), a.obs != nullptr);
        } else {
            t.M[lane] = 0ull;
        }
    }
    __syncthreads();
    // phase 2: the block's warps expand the rows
    emit_block<EPW, OBS>(t, (int)threadIdx.x, (int)blockDim.x, env_base, n_valid, a.obs, a.mask, a.mask_vec);
}

// check mode: replay the whole auction of trajectory i (one thread each)
__global__ void __launch_bounds__(256) k_sl_check(const SlArgs a) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const int64_t off = a.offsets[i], n_calls = a.offsets[i + 1] - off;
    Env e;
    sl_reset(e, (uint32_t)i);
    uint8_t st = BRL_SL_OK;
    for (int64_t k = 0; k < n_calls && st == BRL_SL_OK; ++k) {
        const int32_t c = (int32_t)a.calls[off + k];
        if (f_terminated(e)) st = BRL_SL_EARLY_END;
        else if (c >= kNumActions || !((env_legal_mask(e) >> c) & 1ull)) st = BRL_SL_ILLEGAL;
        else env_step(e, c, TableRows{a.table}, -1.0f, 1.0f);
    }
    if (st == BRL_SL_OK && !f_terminated(e)) st = BRL_SL_NOT_ENDED;
    a.status[i] = st;
}

template <int EPW, int OBS>
static void launch_sl_examples_inst(const SlArgs& a, cudaStream_t s) {
    const unsigned grid = (unsigned)((a.n + EPW - 1) / EPW);
    k_sl_examples<EPW, OBS><<<grid, 128, sizeof(WarpTile<EPW>), s>>>(a);
}
template <int OBS>
static void launch_sl_examples_obs(const SlArgs& a, cudaStream_t s) {
    // 8 examples per block below 65,536 (enough blocks for every SM at B = 10,000), 16 above (not tuned)
    if (a.n < 65536) launch_sl_examples_inst<8, OBS>(a, s);
    else launch_sl_examples_inst<16, OBS>(a, s);
}

}  // namespace brl

extern "C" {

int32_t brl_sl_examples(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;
    const bool check = (p->flags & BRL_F_SL_CHECK) != 0;
    if (p->n_deals <= 0) return fail(BRL_E_OPAQUE, "brl_sl_examples: n_deals must be the number of trajectories (> 0)");
    static const char* names[] = {"deal_table", "calls", "offsets", "traj", "position", "obs", "mask", "label", "position_out", "status"};
    for (int k : {0, 1, 2})
        if (b[k] == nullptr) return fail(BRL_E_BUFFER, "brl_sl_examples: buffer '%s' is NULL", names[k]);
    if (reinterpret_cast<uintptr_t>(b[0]) & 15u) return fail(BRL_E_BUFFER, "brl_sl_examples: buffer 'deal_table' is not 16-byte aligned");
    SlArgs a{};
    a.table = static_cast<const uint8_t*>(b[0]);
    a.calls = static_cast<const uint8_t*>(b[1]);
    a.offsets = static_cast<const int64_t*>(b[2]);
    a.n = p->n_envs;
    a.n_traj = p->n_deals;
    a.env_offset = p->env_offset;
    a.seed = p->seed;
    a.step = p->step;
    cudaStream_t s = (cudaStream_t)stream;
    if (check) {
        if (b[9] == nullptr) return fail(BRL_E_BUFFER, "brl_sl_examples: buffer 'status' is NULL");
        if (a.n > a.n_traj) return fail(BRL_E_OPAQUE, "brl_sl_examples: check mode covers n_envs <= n_deals trajectories");
        a.status = static_cast<uint8_t*>(b[9]);
        k_sl_check<<<(unsigned)((a.n + 255) / 256), 256, 0, s>>>(a);
        return check_launch("brl_sl_examples (check)");
    }
    for (int k : {3, 5, 6, 7})
        if (b[k] == nullptr) return fail(BRL_E_BUFFER, "brl_sl_examples: buffer '%s' is NULL", names[k]);
    if (reinterpret_cast<uintptr_t>(b[5]) & 15u) return fail(BRL_E_BUFFER, "brl_sl_examples: buffer 'obs' is not 16-byte aligned");
    a.traj = static_cast<const int32_t*>(b[3]);
    a.position = static_cast<const int32_t*>(b[4]);
    a.obs = b[5];
    a.mask = static_cast<uint8_t*>(b[6]);
    a.label = static_cast<int32_t*>(b[7]);
    a.position_out = static_cast<int32_t*>(b[8]);
    a.mask_vec = (reinterpret_cast<uintptr_t>(b[6]) & 15u) == 0;  // one row per example: the run of a tile starts at 16 B
    if (p->flags & BRL_F_OBS_U8) launch_sl_examples_obs<kObsU8>(a, s);
    else if (p->flags & BRL_F_OBS_BF16) launch_sl_examples_obs<kObsBF16>(a, s);
    else launch_sl_examples_obs<kObsF32>(a, s);
    return check_launch("brl_sl_examples");
}

}  // extern "C"
