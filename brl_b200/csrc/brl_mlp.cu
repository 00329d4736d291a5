// brl_mlp.cu -- the policy/value net of the rollout and evaluation loops on the 5th-gen
// tensor cores: the "DeepMind" 480 -> 4 x 1024 ReLU -> {38 logits, 1 value} MLP
// (src/models.py:23-33) on TMA + tcgen05 GEMM tiles.  sm_100a only.
//
// The reference runs this net in fp32 (haiku default).  A single bf16 product would
// change near-tie argmax decisions, so the default mode here is a THREE-TERM bf16 split
//     x . w  ~=  x_hi . w_hi  +  x_lo . w_hi  +  x_hi . w_lo        (hi = bf16(v), lo = bf16(v - hi))
// accumulated in fp32 in tensor memory: ~2^-16 relative error per product, i.e. fp32-class
// results at 1/3 of the bf16 tensor rate (still ~6x the fp32 SIMT GEMM rate).  The first
// layer's input is the 0/1 observation, exact in bf16, so it needs only two terms.
// BRL_F_MLP_BF16 selects the plain single-product mode.
//
// Two forward paths, chosen by batch size (fused_forward): below kPairMinM = 4096 rows, five launches of k_mlp_layer;
// from 4096 rows on, one persistent launch of k_mlp_fused for the whole net.
//
// k_mlp_layer, one layer per launch: C[M, N] = act(A[M, K] . Wt[N, K]^T + b).
//   Persistent, one CTA per SM; CTA tile 128 (envs) x BN (features), K in blocks of 64 bf16 = one 128-byte
//   swizzle row; two TMEM accumulators so the epilogue of one tile overlaps the main loop of the next.
//   warp 0    TMA producer: per K block, bulk-tensor loads of the A / Wt (hi, lo) boxes into a
//             ring of shared-memory stages (128B swizzle), completion on an mbarrier;
//   warp 1    MMA issuer: one lane issues tcgen05.mma (UMMA 128 x BN x 16, kind::f16, fp32
//             accumulate in TMEM); tcgen05.commit hands the stage back / signals the epilogue;
//   warps 2-5 epilogue: tcgen05.ld the accumulator (thread = one env row), + bias, ReLU,
//             split into bf16 hi / lo for the next layer (or fp32 logits + value for the head).
// k_mlp_fused, all five layers in one launch: the same roles on CTA pairs (cta_group::2, 256-row tiles), with every
//   layer's tiles in one list and per-row-block counters in place of the launch boundaries between layers.
#include <cuda.h>
#include <cuda_bf16.h>

#include <type_traits>

#include "common.h"
#include "env_device.cuh"
#include "mlp_device.cuh"

namespace brl {

// w[in, out] fp32 (haiku layout, y = x @ w + b) -> Wt_hi / Wt_lo [out_pad, in] bf16 (K-major rows)
__global__ void __launch_bounds__(256) k_mlp_pack(const float* __restrict__ w, const float* __restrict__ b,
                                                  const float* __restrict__ w2, const float* __restrict__ b2,
                                                  __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo,
                                                  float* __restrict__ bias, int k_in, int n_out, int n_src, int n_src2) {
    // rows [0, n_src) come from w, rows [n_src, n_src + n_src2) from w2 (the value head), the rest are zero
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)n_out * k_in) return;
    int n = (int)(idx / k_in), k = (int)(idx % k_in);
    float v = 0.0f;
    if (n < n_src) v = w[(size_t)k * n_src + n];
    else if (n < n_src + n_src2) v = w2[(size_t)k * n_src2 + (n - n_src)];
    __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[idx] = h;
    lo[idx] = __float2bfloat16_rn(v - __bfloat162float(h));
    if (k == 0) bias[n] = n < n_src ? b[n] : (n < n_src + n_src2 ? b2[n - n_src] : 0.0f);
}

// observation f32 / u8 (0/1) -> bf16, for callers whose env emits the reference dtypes
template <class T>
__global__ void __launch_bounds__(256) k_obs_to_bf16(const T* __restrict__ in, __nv_bfloat16* __restrict__ out, int64_t n) {
    int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
    if (i >= n) return;
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        uint32_t a = (float)in[i + 2 * k] != 0.0f ? 0x3F80u : 0u, c = (float)in[i + 2 * k + 1] != 0.0f ? 0x3F80u : 0u;
        w[k] = a | (c << 16);
    }
    *reinterpret_cast<uint4*>(out + i) = make_uint4(w[0], w[1], w[2], w[3]);
}


// ---- epilogues: thread = one env row of the accumulator (TMEM lane), shared by all layer kernels ----------
// hidden layer: + bias, ReLU, split into bf16 hi / lo for the next layer (128-bit stores)
#ifdef BRL_MLP_TRACE
__device__ unsigned long long g_mlp_epi[4];  // debug: SM clocks warp 2 spent in {tcgen05.ld + wait, arithmetic, stores, chunks}
#define BRL_EPI_T0() long long _e0 = clock64()
#define BRL_EPI_ACC(k) do { long long _e1 = clock64(); if ((threadIdx.x & 31) == 0 && (threadIdx.x >> 5) == 2 && blockIdx.x == 0) atomicAdd(&g_mlp_epi[k], (unsigned long long)(_e1 - _e0)); _e0 = _e1; } while (0)
#else
#define BRL_EPI_T0()
#define BRL_EPI_ACC(k)
#endif

// SMEM_BIAS: `bias` points into shared memory (the fused forward stages every layer's bias once per CTA: with ~194 KB of the
// SM given to the operand ring, what is left of L1 does not keep the 4 KB bias vector against the tile's own 131 KB of
// stores, and 16 global loads per 32-column chunk each waited a full L2 round trip -- scripts/exp_mlp_trace.py)
template <bool SMEM_BIAS = false>
__device__ __forceinline__ void epilogue_hidden_row(uint32_t t_row, int n_cols, const float* __restrict__ bias, bool row_ok,
                                                    __nv_bfloat16* __restrict__ out_hi, __nv_bfloat16* __restrict__ out_lo) {
    BRL_EPI_T0();
#pragma unroll 1
    for (int c0 = 0; c0 < n_cols; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(t_row + (uint32_t)c0, r);
        BRL_EPI_ACC(0);
        if (row_ok) {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
                const float2 bb = SMEM_BIAS ? reinterpret_cast<const float2*>(bias + c0)[jj]
                                            : __ldg(reinterpret_cast<const float2*>(bias + c0) + jj);  // warp-uniform
                float x0 = fmaxf(__uint_as_float(r[2 * jj]) + bb.x, 0.0f);
                float x1 = fmaxf(__uint_as_float(r[2 * jj + 1]) + bb.y, 0.0f);
                __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
                hi[jj] = *reinterpret_cast<uint32_t*>(&h);
                lo[jj] = pack_bf16x2(x0 - __low2float(h), x1 - __high2float(h));
            }
            BRL_EPI_ACC(1);
            uint4* ph = reinterpret_cast<uint4*>(out_hi + c0);
#pragma unroll
            for (int v = 0; v < 4; ++v) ph[v] = make_uint4(hi[4 * v], hi[4 * v + 1], hi[4 * v + 2], hi[4 * v + 3]);
            if (out_lo) {
                uint4* pl = reinterpret_cast<uint4*>(out_lo + c0);
#pragma unroll
                for (int v = 0; v < 4; ++v) pl[v] = make_uint4(lo[4 * v], lo[4 * v + 1], lo[4 * v + 2], lo[4 * v + 3]);
            }
            BRL_EPI_ACC(2);
        }
    }
}

// Hidden-layer epilogue of the fused forward with TMA stores.  A thread owns one accumulator row; written straight to global
// memory its 16-byte pieces land in 32 different rows per warp instruction (32 LSU wavefronts each, 8192 per 128 x 256
// tile: ~4 us of the SM's load/store pipe -- the epilogue took 10-12 us per tile, longer than layer 0's 6 us main loop and on
// every layer's dependency path, scripts/exp_mlp_trace.py).  Here each 32-column chunk is staged in shared memory as the
// 32-row x 64-byte box of a 64B-swizzled tensor map (lane = row, conflict-free 128-bit stores) and one lane issues a bulk
// tensor store for the hi and the lo block; rows past M are clipped by the map.  `stage` = this warp's 2 x 2 KB.
__device__ __forceinline__ void epilogue_hidden_tma(uint32_t t_row, int n_cols, const float* __restrict__ bias, int lane,
                                                    uint32_t stage, const CUtensorMap* st_hi, const CUtensorMap* st_lo,
                                                    int col0, int row0) {
    BRL_EPI_T0();
    const uint32_t sw = (uint32_t)((lane >> 1) & 3);  // 64B swizzle: 16-byte chunk index ^= bits 7-8 of the byte offset
#pragma unroll 1
    for (int c0 = 0; c0 < n_cols; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(t_row + (uint32_t)c0, r);
        BRL_EPI_ACC(0);
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) {
            const float2 bb = __ldg(reinterpret_cast<const float2*>(bias + c0) + jj);  // warp-uniform
            float x0 = fmaxf(__uint_as_float(r[2 * jj]) + bb.x, 0.0f);
            float x1 = fmaxf(__uint_as_float(r[2 * jj + 1]) + bb.y, 0.0f);
            __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
            hi[jj] = *reinterpret_cast<uint32_t*>(&h);
            lo[jj] = pack_bf16x2(x0 - __low2float(h), x1 - __high2float(h));
        }
        BRL_EPI_ACC(1);
        if (c0 > 0) {  // the previous chunk's stores have read the staging blocks
            if (lane == 0) bulk_wait_read0();
            __syncwarp();
        }
        const uint32_t row_hi = stage + (uint32_t)lane * 64u, row_lo = row_hi + 2048u;
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            const uint32_t off = ((uint32_t)v ^ sw) * 16u;
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row_hi + off), "r"(hi[4 * v]), "r"(hi[4 * v + 1]),
                         "r"(hi[4 * v + 2]), "r"(hi[4 * v + 3]) : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row_lo + off), "r"(lo[4 * v]), "r"(lo[4 * v + 1]),
                         "r"(lo[4 * v + 2]), "r"(lo[4 * v + 3]) : "memory");
        }
        fence_async_smem();  // generic-proxy writes -> async-proxy (TMA) reads
        __syncwarp();
        if (lane == 0) {
            tma_store_2d(st_hi, stage, col0 + c0, row0);
            tma_store_2d(st_lo, stage + 2048u, col0 + c0, row0);
            bulk_commit();
        }
        BRL_EPI_ACC(2);
    }
}

// head tile with the masked categorical of src/roll_out.py:27-30,79-81 fused in: the thread that owns an env row
// holds its 38 logits in registers, so where(mask, logits, -inf), the Gumbel-argmax sample (same Philox stream as
// brl_categorical: counter (env, GUM0 + a / 4, step), key = seed) or the first-argmax mode, and
// log_softmax(masked)[action] cost no extra launch and no logits round trip.
struct ActArgs {
    const uint8_t* mask;   // [n, 38] or NULL (unmasked)
    int32_t* action;       // [n]; NULL = no categorical fused (plain forward)
    float* log_prob;       // [n] or NULL
    uint64_t seed;
    int64_t env_offset;
    uint32_t step;
    int sample;
    const int32_t* row_index;  // [n] or NULL: row r of the batch is env row_index[r] (mask / action / log_prob / value / RNG by env)
    const uint64_t* seed_salt; // device u64 or NULL: XORed into `seed` (a captured CUDA graph replays with fresh noise)
};

__device__ __forceinline__ void epilogue_head_act_row(uint32_t t_row, const float* __restrict__ bias, bool row_ok, int64_t row,
                                                      float* __restrict__ logits, float* __restrict__ value, const ActArgs& act) {
    uint32_t r0[32], r1[32];
    tmem_ld32(t_row, r0);
    tmem_ld32(t_row + 32u, r1);
    if (!row_ok) return;
    float l[40];
#pragma unroll
    for (int k = 0; k < 32; ++k) l[k] = __uint_as_float(r0[k]) + __ldg(bias + k);
#pragma unroll
    for (int k = 0; k < 7; ++k) l[32 + k] = __uint_as_float(r1[k]) + __ldg(bias + 32 + k);
    l[39] = 0.0f;
    if (act.row_index) row = act.row_index[row];  // a listed batch: every per-env array below is addressed by env
    if (logits) {
        float2* pl = reinterpret_cast<float2*>(logits + row * 38);
#pragma unroll
        for (int jj = 0; jj < 19; ++jj) pl[jj] = make_float2(l[2 * jj], l[2 * jj + 1]);
    }
    if (value) value[row] = l[38];
    if (act.action == nullptr) return;
    uint64_t legal = ~0ull;
    if (act.mask) {
        const uint16_t* pm = reinterpret_cast<const uint16_t*>(act.mask + row * 38);  // 38 * row is even
        legal = 0;
#pragma unroll
        for (int jj = 0; jj < 19; ++jj) {
            const uint32_t m2 = pm[jj];
            legal |= (uint64_t)((m2 & 0xFFu) != 0) << (2 * jj) | (uint64_t)((m2 >> 8) != 0) << (2 * jj + 1);
        }
    }
    const uint64_t g = (uint64_t)(act.env_offset + row);
    const uint64_t seed = act.seed_salt ? (act.seed ^ __ldg(act.seed_salt)) : act.seed;
    float best = -INFINITY, mx = -INFINITY, la = 0.0f;
    int best_a = kNumActions;
#pragma unroll
    for (int grp = 0; grp < 10; ++grp) {
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        if (act.sample) {
            const uint4 rr = philox4x32(make_uint4((uint32_t)g, (uint32_t)(g >> 32), kTagGum + (uint32_t)grp, act.step),
                                        make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
            w[0] = rr.x; w[1] = rr.y; w[2] = rr.z; w[3] = rr.w;
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int aidx = 4 * grp + e;
            if (aidx < kNumActions && ((legal >> aidx) & 1ull)) {
                float v = l[aidx];
                if (act.sample) {
                    const float u = ((float)(w[e] >> 8) + 0.5f) * (1.0f / 16777216.0f);
                    v += -logf(-logf(u));
                }
                if (v > best) { best = v; best_a = aidx; la = l[aidx]; }  // ascending: ties keep the lower index
                mx = fmaxf(mx, l[aidx]);
            }
        }
    }
    float se = 0.0f;
#pragma unroll
    for (int aidx = 0; aidx < kNumActions; ++aidx)
        if ((legal >> aidx) & 1ull) se += expf(l[aidx] - mx);
    if (best_a >= kNumActions) { best_a = 0; la = l[0]; }  // no legal action: cannot happen for a valid mask
    act.action[row] = best_a;
    if (act.log_prob) act.log_prob[row] = la - mx - logf(se);
}

// ---- one layer ------------------------------------------------------------------------------
struct LayerArgs {
    const float* bias;           // [n_pad]
    __nv_bfloat16* out_hi;       // hidden: [M, n_total] bf16
    __nv_bfloat16* out_lo;       // hidden, split mode: residual (may be NULL)
    float* logits;               // head: [M, 38]
    float* value;                // head: [M]
    int M, n_total, k_blocks;
    int n_tiles_n, n_tiles;      // tiles along N, total tiles of this layer
};
// grouped forward (a pool of nets): rows [b * kGroupRows, (b + 1) * kGroupRows) use model block_model[b]; the pool's biases are
// bias_stride floats apart; the grouped head runs the masked argmax of `act` in its epilogue.  The row count is read from device
// memory: the launch and its tensor maps are sized for the grouping's capacity, and the row blocks past the count exit at once.
// A separate type, so that the ungrouped kernels keep their parameter block (and their code) as it was.
struct GroupedLayerArgs : LayerArgs {
    const int32_t* block_model;
    int64_t bias_stride;
    ActArgs act;
    const int32_t* n_rows;  // padded row count (brl_model_rows' offsets[M])
};
template <bool GROUPED>
using LayerArgsT = std::conditional_t<GROUPED, GroupedLayerArgs, LayerArgs>;
__device__ __forceinline__ int layer_rows(const LayerArgs& a) { return a.M; }
__device__ __forceinline__ int layer_rows(const GroupedLayerArgs& a) { return *a.n_rows; }
__device__ __forceinline__ int layer_tiles(const LayerArgs& a) { return a.n_tiles; }
__device__ __forceinline__ int layer_tiles(const GroupedLayerArgs& a) { return a.n_tiles_n * ((*a.n_rows + kBM - 1) / kBM); }

template <int BN, bool SPLIT_A, bool SPLIT_W>
struct LayerCfg {
    static constexpr uint32_t kABytes = kBM * kBK * 2, kWBytes = BN * kBK * 2;
    static constexpr uint32_t kStageBytes = kABytes * (SPLIT_A ? 2 : 1) + kWBytes * (SPLIT_W ? 2 : 1);
    static constexpr int kStages = (kSmemBudget / kStageBytes) > 8 ? 8 : (int)(kSmemBudget / kStageBytes);
    static constexpr uint32_t kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/;
};

template <int BN, bool SPLIT_A, bool SPLIT_W, bool HEAD, bool GROUPED = false>
__global__ void __launch_bounds__(kMlpThreads, 1)
k_mlp_layer(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
            const __grid_constant__ CUtensorMap tm_w_hi, const __grid_constant__ CUtensorMap tm_w_lo,
            const LayerArgsT<GROUPED> a) {
    // PERSISTENT: one CTA per SM walks tiles blockIdx.x, blockIdx.x + gridDim.x, ... (n-tile fastest, so the
    // CTAs running together share A row-blocks in L2).  The smem stage ring runs straight across tile
    // boundaries and the accumulator is double-buffered in TMEM, so the epilogue of tile j overlaps the
    // TMA + MMA main loop of tile j + 1.
    using Cfg = LayerCfg<BN, SPLIT_A, SPLIT_W>;
    constexpr int S = Cfg::kStages;
    constexpr uint32_t kTmemCols = 2 * BN;  // two accumulators of BN fp32 columns (power of two >= 32)
    extern __shared__ unsigned char smem_dyn[];
    const uint32_t base = (smem_addr(smem_dyn) + 1023u) & ~1023u;  // 128B swizzle atoms need 1024-byte alignment
    const uint32_t bar_base = base + S * Cfg::kStageBytes;         // full[S], empty[S], tmem_full[2], tmem_empty[2]
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (S + s); };
    auto tmem_full_bar = [&](int b) { return bar_base + 8u * (2 * S + b); };
    auto tmem_empty_bar = [&](int b) { return bar_base + 8u * (2 * S + 2 + b); };
    __shared__ uint32_t tmem_base_s;  // written by tcgen05.alloc

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_tiles_n = a.n_tiles_n, n_tiles = layer_tiles(a);

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_a_hi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_w_hi) : "memory");
        if (SPLIT_A) asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_a_lo) : "memory");
        if (SPLIT_W) asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_w_lo) : "memory");
        for (int s = 0; s < S; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(tmem_full_bar(b), 1); mbar_init(tmem_empty_bar(b), 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_addr(&tmem_base_s), kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_acc = *reinterpret_cast<volatile uint32_t*>(&tmem_base_s);

    if (warp == 0) {
        if (lane == 0) {  // ===== TMA producer =====
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const int m0 = (tile / n_tiles_n) * kBM, n0 = (tile % n_tiles_n) * BN;
                int model = 0;
                if constexpr (GROUPED) model = a.block_model[m0 / kGroupRows];
                for (int kb = 0; kb < a.k_blocks; ++kb, ++it) {
                    const int s = (int)(it % S);
                    mbar_wait(empty_bar(s), ((it / S) & 1u) ^ 1u);
                    mbar_expect_tx(full_bar(s), Cfg::kStageBytes);
                    uint32_t dst = base + s * Cfg::kStageBytes;
                    tma_load_2d(dst, &tm_a_hi, full_bar(s), kb * kBK, m0);
                    dst += Cfg::kABytes;
                    if (SPLIT_A) { tma_load_2d(dst, &tm_a_lo, full_bar(s), kb * kBK, m0); dst += Cfg::kABytes; }
                    if constexpr (GROUPED) {  // the pool's weights as {k, n, model}: this row block's net
                        tma_load_3d(dst, &tm_w_hi, full_bar(s), kb * kBK, n0, model);
                        if (SPLIT_W) tma_load_3d(dst + Cfg::kWBytes, &tm_w_lo, full_bar(s), kb * kBK, n0, model);
                    } else {
                        tma_load_2d(dst, &tm_w_hi, full_bar(s), kb * kBK, n0);
                        dst += Cfg::kWBytes;
                        if (SPLIT_W) tma_load_2d(dst, &tm_w_lo, full_bar(s), kb * kBK, n0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {  // ===== MMA issuer =====
            constexpr uint32_t idesc = umma_idesc_bf16(kBM, BN);
            uint32_t it = 0, j = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++j) {
                const uint32_t buf = j & 1u;
                mbar_wait(tmem_empty_bar(buf), ((j >> 1) & 1u) ^ 1u);  // the epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t acc = tmem_acc + buf * BN;
                for (int kb = 0; kb < a.k_blocks; ++kb, ++it) {
                    const int s = (int)(it % S);
                    mbar_wait(full_bar(s), (it / S) & 1u);
                    tc_fence_after();
                    const uint32_t sa_hi = base + s * Cfg::kStageBytes;
                    const uint32_t sa_lo = sa_hi + Cfg::kABytes;
                    const uint32_t sw_hi = sa_hi + Cfg::kABytes * (SPLIT_A ? 2 : 1);
                    const uint32_t sw_lo = sw_hi + Cfg::kWBytes;
#pragma unroll
                    for (int k = 0; k < kBK / kUmmaK; ++k) {
                        const uint32_t koff = (uint32_t)k * kUmmaK * 2;  // bytes along K inside the 128-byte row
                        const uint64_t da_hi = umma_desc_sw128(sa_hi + koff), dw_hi = umma_desc_sw128(sw_hi + koff);
                        umma_bf16(acc, da_hi, dw_hi, idesc, (kb | k) != 0);
                        if (SPLIT_A) umma_bf16(acc, umma_desc_sw128(sa_lo + koff), dw_hi, idesc, 1u);
                        if (SPLIT_W) umma_bf16(acc, da_hi, umma_desc_sw128(sw_lo + koff), idesc, 1u);
                    }
                    umma_commit(empty_bar(s));  // the stage is free once these MMAs have read it
                }
                umma_commit(tmem_full_bar(buf));
            }
        }
    } else {  // ===== epilogue: warps 2..5, TMEM lane quarter = warp % 4 =====
        const int q = warp & 3, M = layer_rows(a);
        uint32_t j = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++j) {
            const int m0 = (tile / n_tiles_n) * kBM, n0 = (tile % n_tiles_n) * BN;
            const uint32_t buf = j & 1u;
            mbar_wait(tmem_full_bar(buf), (j >> 1) & 1u);
            tc_fence_after();
            const int row = m0 + q * 32 + lane;
            const uint32_t t_row = tmem_acc + buf * BN + ((uint32_t)(q * 32) << 16);
            const float* bias = a.bias + n0;
            if constexpr (GROUPED) bias += (size_t)a.block_model[m0 / kGroupRows] * a.bias_stride;
            if constexpr (!HEAD)
                epilogue_hidden_row(t_row, BN, bias, row < M, a.out_hi + (size_t)row * a.n_total + n0,
                                    a.out_lo ? a.out_lo + (size_t)row * a.n_total + n0 : nullptr);
            else if constexpr (GROUPED)  // padding rows of a group (row_index -1) are computed and dropped
                epilogue_head_act_row(t_row, bias, row < M && a.act.row_index[row] >= 0, row, a.logits, nullptr, a.act);
            else
                epilogue_head_row(t_row, bias, row < M, a.logits + (size_t)row * 38, a.value + row);
            // all of this warp's tcgen05.ld have completed (wait::ld): hand the accumulator back
            tc_fence_before();
            __syncwarp();
            if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tmem_empty_bar(buf)) : "memory");
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_acc, kTmemCols);
}

// ---- CTA pairs (cta_group::2): the tiles of k_mlp_fused -----------------------------------------
// The 1-CTA tiles above are bound by the L2 -> SM operand fill (~64 B/clk/SM against the split mode's
// 83 B/clk demand at 128 x 128).  A CTA pair (cluster of 2 = the two SMs of a TPC) computes a 256 x BN tile
// with ONE tcgen05.mma.cta_group::2 stream issued by the leader: each CTA stages its own 128 env rows of A and
// only HALF of the Wt rows (the MMA reads the other half out of the peer's shared memory), and accumulates its
// own 128 x BN block in its own TMEM.  Operand bytes per MMA clock: 42 B/clk/SM at BN = 256.
//   full[s]        lives in the leader; both CTAs' TMA loads complete_tx on it (cta_group::2, peer bit masked);
//   empty[s]       one per CTA, released by the leader's multicast tcgen05.commit;
//   tmem_full[b]   one per CTA, multicast commit;   tmem_empty[b]  in the leader, 16 arrivals (8 epilogue warps x 2 CTAs).
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;  // shared::cluster address of the same offset in the pair's even CTA

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d_pair(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {  // arrives on `bar`'s offset in BOTH CTAs
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
}

// ---- the whole forward as ONE persistent launch on CTA pairs ----------------------------------------
// Five separate launches lose (i) a wave-quantisation tail per layer (8192 envs = 128 pair tiles on 74 pairs =
// 1.73 waves) and (ii) the drain / launch / pipeline-fill gap between layers.  Here all 4 x 128 + 32 tiles of the
// five layers form one list, walked round-robin by the persistent pairs; a tile of layer l + 1 needs only the
// 128-row block of layer l's output it reads, so the next layer's first tiles fill the previous layer's tail.
// Dependency tracking: every epilogue warp publishes (st.global ... fence, red.add) into ready[l][128-row block];
// the TMA producer acquires the count (16 = 4 n-tiles x 4 warps) and crosses into the async proxy before its
// first A load of the tile.  Tiles are claimed in list order and depend only on earlier tiles, and the grid never
// exceeds the co-resident cluster count, so the waits cannot deadlock (spins are bounded: a bug traps).
struct FusedArgs {
    CUtensorMap a_hi[5], a_lo[5], w_hi[5], w_lo[5];
    CUtensorMap st_hi[4], st_lo[4];  // the hidden layers' outputs as TMA-store destinations (32 x 32 boxes)
    const float* bias[5];
    __nv_bfloat16* out_hi[4];
    __nv_bfloat16* out_lo[4];
    float* logits;
    float* value;
    uint32_t* ready;  // [4][2 * nmb], zeroed before the launch
    int M, nmb, tiles_per_layer, n_tiles;
    ActArgs act;
};
struct GroupedFusedArgs : FusedArgs {  // grouped forward (see GroupedLayerArgs): M, nmb and the tile list follow *n_rows
    const int32_t* block_model;  // model of each kGroupRows-row block (= the CTA-pair tile height)
    int64_t bias_stride;         // floats between two nets' biases in the pool
    const int32_t* n_rows;
};
template <bool GROUPED>
using FusedArgsT = std::conditional_t<GROUPED, GroupedFusedArgs, FusedArgs>;

constexpr int kFusedBN = 256, kFusedTilesN = kHidden / kFusedBN;
// Epilogue warps of the fused forward: TWO per TMEM lane quadrant, each draining half of the tile's 256 columns.  One
// warp per quadrant sits alone on its SM sub-partition and runs the bias / ReLU / bf16-split chain at ~7 clocks per
// instruction (scripts/exp_mlp_trace.py: 10-12 us per tile, longer than layer 0's 6 us main loop and on every layer's
// dependency path); two warps of a quadrant share a sub-partition and interleave.
constexpr int kFusedEpiWarps = 8, kFusedThreads = 32 * (2 + kFusedEpiWarps);
constexpr uint32_t kReadyPerBlock = kFusedTilesN * kFusedEpiWarps;  // n-tiles x epilogue warps

template <bool SPLIT>
struct FusedCfg {
    static constexpr uint32_t kABytes = kBM * kBK * 2, kWBytes = (kFusedBN / 2) * kBK * 2, kWHeadBytes = (kHeadPad / 2) * kBK * 2;
    static constexpr uint32_t kStageBytes = (kABytes + kWBytes) * (SPLIT ? 2 : 1);
    static constexpr int kStages = (kSmemBudget / kStageBytes) > 8 ? 8 : (int)(kSmemBudget / kStageBytes);
    static constexpr uint32_t kStoreStageBytes = 8 /*epilogue warps*/ * 2 /*hi, lo*/ * 2048;  // 32 rows x 64 B per warp and array
    static constexpr uint32_t kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/ + 1024 /*align*/ + kStoreStageBytes;
    static_assert(kSmemBytes <= 227 * 1024, "operand ring + store staging exceed the SM's shared memory");
};

struct FusedTile { int layer, mb, nt; };
__device__ __forceinline__ FusedTile fused_tile(int t, int tiles_per_layer) {
    FusedTile f;
    f.layer = t / tiles_per_layer;
    if (f.layer < 4) {
        const int r = t - f.layer * tiles_per_layer;
        f.mb = r / kFusedTilesN;
        f.nt = r % kFusedTilesN;
    } else {
        f.layer = 4;
        f.mb = t - 4 * tiles_per_layer;
        f.nt = 0;
    }
    return f;
}

#ifdef BRL_MLP_TRACE
// debug build (scripts/exp_mlp_trace.py): per-tile %globaltimer stamps of the fused forward, written by the leader CTA's role lanes
// [0] dependency wait begins [1] dependency ready [2] last TMA issued [3] accumulator free, first MMA [4] last MMA committed
// [5] accumulator seen by the epilogue [6] tile published [7] pair
__device__ unsigned long long g_mlp_trace[1024][8];
__device__ __forceinline__ unsigned long long mlp_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define BRL_MLP_STAMP(tile, k) do { if (leader && (tile) < 1024) g_mlp_trace[tile][k] = mlp_now(); } while (0)
#else
#define BRL_MLP_STAMP(tile, k)
#endif

// layer `layer`'s bias of row block `mb`'s net, and whether `row` is an env's row (padding rows of a group are dropped)
__device__ __forceinline__ const float* fused_bias(const FusedArgs& a, int layer, int) { return a.bias[layer]; }
__device__ __forceinline__ const float* fused_bias(const GroupedFusedArgs& a, int layer, int mb) {
    return a.bias[layer] + (size_t)a.block_model[mb] * a.bias_stride;
}
__device__ __forceinline__ bool fused_row_ok(const FusedArgs& a, int row) { return row < a.M; }
__device__ __forceinline__ bool fused_row_ok(const GroupedFusedArgs& a, int row) { return row < *a.n_rows && a.act.row_index[row] >= 0; }

// the launch's shape -- rows, 256-row blocks, tiles per hidden layer, tiles -- from the parameters, or (grouped) from *n_rows
__device__ __forceinline__ int fused_rows(const FusedArgs& a) { return a.M; }
__device__ __forceinline__ int fused_rows(const GroupedFusedArgs& a) { return *a.n_rows; }
__device__ __forceinline__ int fused_nmb(const FusedArgs& a) { return a.nmb; }
__device__ __forceinline__ int fused_nmb(const GroupedFusedArgs& a) { return (*a.n_rows + 2 * kBM - 1) / (2 * kBM); }
__device__ __forceinline__ int fused_tiles_per_layer(const FusedArgs& a) { return a.tiles_per_layer; }
__device__ __forceinline__ int fused_tiles_per_layer(const GroupedFusedArgs& a) { return fused_nmb(a) * kFusedTilesN; }
__device__ __forceinline__ int fused_n_tiles(const FusedArgs& a) { return a.n_tiles; }
__device__ __forceinline__ int fused_n_tiles(const GroupedFusedArgs& a) { return fused_nmb(a) * (4 * kFusedTilesN + 1); }

template <bool SPLIT, bool GROUPED = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kFusedThreads, 1)
k_mlp_fused(const __grid_constant__ FusedArgsT<GROUPED> a) {
    using Cfg = FusedCfg<SPLIT>;
    constexpr int S = Cfg::kStages;
    constexpr uint32_t kTmemCols = 2 * kFusedBN;
    extern __shared__ unsigned char smem_dyn[];
    const uint32_t base = (smem_addr(smem_dyn) + 1023u) & ~1023u;
    const uint32_t bar_base = base + S * Cfg::kStageBytes;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (S + s); };
    auto tmem_full_bar = [&](int b) { return bar_base + 8u * (2 * S + b); };
    auto tmem_empty_bar = [&](int b) { return bar_base + 8u * (2 * S + 2 + b); };
    const uint32_t store_base = (bar_base + 256u + 1023u) & ~1023u;  // 8 epilogue warps x (hi, lo) x 2 KB store staging
    __shared__ uint32_t tmem_base_s;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
    const int n_tiles = fused_n_tiles(a), tpl = fused_tiles_per_layer(a);

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < S; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(tmem_full_bar(b), 1); mbar_init(tmem_empty_bar(b), 2 * kFusedEpiWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(&tmem_base_s)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_acc = *reinterpret_cast<volatile uint32_t*>(&tmem_base_s);

    if (warp == 0) {
        if (lane == 0) {  // ===== TMA producer (both CTAs) =====
            const uint32_t lead_full0 = full_bar(0) & kPeerBitMask;
            uint32_t it = 0;
            for (int tile = pair; tile < n_tiles; tile += n_pairs) {
                const FusedTile f = fused_tile(tile, tpl);
                const bool split_a = SPLIT && f.layer > 0;  // the 0/1 observation is exact in bf16
                const int k_blocks = f.layer == 0 ? (kObsDimM + kBK - 1) / kBK : kHidden / kBK;
                const uint32_t w_bytes = f.layer == 4 ? Cfg::kWHeadBytes : Cfg::kWBytes;
                const uint32_t tx = Cfg::kABytes * (split_a ? 2u : 1u) + w_bytes * (SPLIT ? 2u : 1u);
                const int m0 = f.mb * (2 * kBM) + (int)rank * kBM;
                const int n0 = f.layer == 4 ? (int)rank * (kHeadPad / 2) : f.nt * kFusedBN + (int)rank * (kFusedBN / 2);
                const CUtensorMap* ma_hi = &a.a_hi[f.layer];
                const CUtensorMap* ma_lo = &a.a_lo[f.layer];
                const CUtensorMap* mw_hi = &a.w_hi[f.layer];
                const CUtensorMap* mw_lo = &a.w_lo[f.layer];
                BRL_MLP_STAMP(tile, 0);
                if (f.layer > 0) {  // the previous layer's rows [m0, m0 + 128) must be complete (all 4 n-tiles)
                    const uint32_t* flag = a.ready + (size_t)(f.layer - 1) * 2 * fused_nmb(a) + 2 * f.mb + rank;
                    uint32_t v = 0;
                    for (uint32_t spin = 0;; ++spin) {
                        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
                        if (v >= kReadyPerBlock) break;
                        if (spin > (1u << 24)) __trap();
                        __nanosleep(64);
                    }
                    asm volatile("fence.proxy.async;" ::: "memory");  // generic-proxy writes -> async-proxy (TMA) reads
                }
                BRL_MLP_STAMP(tile, 1);
                int model = 0;
                if constexpr (GROUPED) model = a.block_model[f.mb];
                for (int kb = 0; kb < k_blocks; ++kb, ++it) {
                    const int s = (int)(it % S);
                    mbar_wait(empty_bar(s), ((it / S) & 1u) ^ 1u);
                    if (leader) mbar_expect_tx(full_bar(s), 2u * tx);
                    const uint32_t fb = lead_full0 + 8u * s;
                    const uint32_t sa = base + s * Cfg::kStageBytes;
                    const uint32_t sw = sa + Cfg::kABytes * (SPLIT ? 2 : 1);
                    tma_load_2d_pair(sa, ma_hi, fb, kb * kBK, m0);
                    if (split_a) tma_load_2d_pair(sa + Cfg::kABytes, ma_lo, fb, kb * kBK, m0);
                    if constexpr (GROUPED) {  // the pool's weights as {k, n, model}: this row block's net
                        tma_load_3d_pair(sw, mw_hi, fb, kb * kBK, n0, model);
                        if (SPLIT) tma_load_3d_pair(sw + Cfg::kWBytes, mw_lo, fb, kb * kBK, n0, model);
                    } else {
                        tma_load_2d_pair(sw, mw_hi, fb, kb * kBK, n0);
                        if (SPLIT) tma_load_2d_pair(sw + Cfg::kWBytes, mw_lo, fb, kb * kBK, n0);
                    }
                }
                BRL_MLP_STAMP(tile, 2);
            }
        }
    } else if (warp == 1) {
        if (leader && lane == 0) {  // ===== MMA issuer =====
            uint32_t it = 0, j = 0;
            for (int tile = pair; tile < n_tiles; tile += n_pairs, ++j) {
                const FusedTile f = fused_tile(tile, tpl);
                const bool split_a = SPLIT && f.layer > 0;
                const int k_blocks = f.layer == 0 ? (kObsDimM + kBK - 1) / kBK : kHidden / kBK;
                const uint32_t idesc = f.layer == 4 ? umma_idesc_bf16(2 * kBM, kHeadPad) : umma_idesc_bf16(2 * kBM, kFusedBN);
                const uint32_t buf = j & 1u;
                mbar_wait(tmem_empty_bar(buf), ((j >> 1) & 1u) ^ 1u);
                tc_fence_after();
                BRL_MLP_STAMP(tile, 3);
                const uint32_t acc = tmem_acc + buf * kFusedBN;
                for (int kb = 0; kb < k_blocks; ++kb, ++it) {
                    const int s = (int)(it % S);
                    mbar_wait(full_bar(s), (it / S) & 1u);
                    tc_fence_after();
                    const uint32_t sa_hi = base + s * Cfg::kStageBytes;
                    const uint32_t sa_lo = sa_hi + Cfg::kABytes;
                    const uint32_t sw_hi = sa_hi + Cfg::kABytes * (SPLIT ? 2 : 1);
                    const uint32_t sw_lo = sw_hi + Cfg::kWBytes;
#pragma unroll
                    for (int k = 0; k < kBK / kUmmaK; ++k) {
                        const uint32_t koff = (uint32_t)k * kUmmaK * 2;
                        const uint64_t da_hi = umma_desc_sw128(sa_hi + koff), dw_hi = umma_desc_sw128(sw_hi + koff);
                        umma_bf16_pair(acc, da_hi, dw_hi, idesc, (kb | k) != 0);
                        if (split_a) umma_bf16_pair(acc, umma_desc_sw128(sa_lo + koff), dw_hi, idesc, 1u);
                        if (SPLIT) umma_bf16_pair(acc, da_hi, umma_desc_sw128(sw_lo + koff), idesc, 1u);
                    }
                    umma_commit_pair(empty_bar(s));
                }
                umma_commit_pair(tmem_full_bar(buf));
                BRL_MLP_STAMP(tile, 4);
            }
        }
    } else {  // ===== epilogue: warp w drains TMEM lane quadrant w % 4, column half (w - 2) / 4 =====
        const int q = warp & 3, half = (warp - 2) >> 2;
        constexpr int kHalfCols = kFusedBN / 2;
        const uint32_t lead_tmem_empty0 = tmem_empty_bar(0) & kPeerBitMask;
        uint32_t j = 0;
        for (int tile = pair; tile < n_tiles; tile += n_pairs, ++j) {
            const FusedTile f = fused_tile(tile, tpl);
            const int m0 = f.mb * (2 * kBM) + (int)rank * kBM;
            const uint32_t buf = j & 1u;
            mbar_wait(tmem_full_bar(buf), (j >> 1) & 1u);
            tc_fence_after();
            if (warp == 2 && lane == 0) { BRL_MLP_STAMP(tile, 5); }
            const int row = m0 + q * 32 + lane;
            const uint32_t t_row = tmem_acc + buf * kFusedBN + ((uint32_t)(q * 32) << 16);
            if (f.layer < 4) {
                const int n0 = f.nt * kFusedBN + half * kHalfCols;
                if (SPLIT) {
                    epilogue_hidden_tma(t_row + (uint32_t)(half * kHalfCols), kHalfCols, fused_bias(a, f.layer, f.mb) + n0, lane,
                                        store_base + (uint32_t)(warp - 2) * 4096u, &a.st_hi[f.layer], &a.st_lo[f.layer], n0,
                                        m0 + q * 32);
                } else {
                    __nv_bfloat16* oh = a.out_hi[f.layer];
                    epilogue_hidden_row(t_row + (uint32_t)(half * kHalfCols), kHalfCols, fused_bias(a, f.layer, f.mb) + n0, row < fused_rows(a),
                                        oh + (size_t)row * kHidden + n0, nullptr);
                }
            } else if (half == 0) {  // the 64-column head tile: one warp per quadrant
                epilogue_head_act_row(t_row, fused_bias(a, 4, f.mb), fused_row_ok(a, row), row, a.logits, a.value, a.act);
            }
            tc_fence_before();
            __syncwarp();  // orders the other lanes' activation stores before lane 0's fence (sync, one fence, one atomic)
            if (lane == 0) {
                asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(lead_tmem_empty0 + 8u * buf) : "memory");
                if (f.layer < 4) {
                    if (SPLIT) {  // this warp's bulk tensor stores are performed (not just read) before the rows are published
                        bulk_wait0();
                        asm volatile("fence.proxy.async;" ::: "memory");
                    }
                    __threadfence();  // cumulative: the warp's rows are visible GPU-wide before the count below
                    atomicAdd(a.ready + (size_t)f.layer * 2 * fused_nmb(a) + 2 * f.mb + rank, 1u);
                }
#ifdef BRL_MLP_TRACE
                if (warp == 2 && leader && tile < 1024) { g_mlp_trace[tile][6] = mlp_now(); g_mlp_trace[tile][7] = (unsigned long long)pair; }
#endif
            }
        }
    }
    tc_fence_before();
    cluster_sync_all();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"(kTmemCols) : "memory");
}


// a pool of nets (brl_policy_act_grouped): `n_models` packed blobs `stride` bytes apart, and the model of each kGroupRows-row block
struct PoolArgs {
    const int32_t* block_model;
    int64_t stride;
    int n_models;
    ActArgs act;  // the per-layer head's masked argmax (the fused head takes launch_fused's `act`)
    const int32_t* n_rows;  // the padded row count in device memory (the launch is sized for M = the capacity)
};

// weight operand of layer-tile loads: one net's [n_rows, k_in] bf16 matrix, or the pool's {k_in, n_rows, model} stack of them
template <bool GROUPED>
static bool make_w_map(CUtensorMap* m, const void* w, uint64_t n_rows, uint64_t k_in, uint32_t box_rows, const PoolArgs* pool) {
    if constexpr (!GROUPED) return make_map(m, w, n_rows, k_in, k_in, box_rows);
    const uint64_t dims[3] = {k_in, n_rows, (uint64_t)pool->n_models}, strides[2] = {k_in * 2, (uint64_t)pool->stride};
    const uint32_t box[3] = {(uint32_t)kBK, box_rows, 1};
    return make_map_nd(m, w, 3, dims, strides, box);
}

// the kernel's shared-memory attribute, set once per device (idempotent, a race only repeats the call); also called ahead of a
// stream capture (brl_duplicate_match) so that no attribute call falls inside one
template <int BN, bool SPLIT_A, bool SPLIT_W, bool HEAD, bool GROUPED = false>
static int32_t layer_attr() {
    using Cfg = LayerCfg<BN, SPLIT_A, SPLIT_W>;
    static bool attr_set_dev[kMaxDevices] = {};
    bool& attr_set = attr_set_dev[device_slot()];
    if (!attr_set) {
        if (cudaFuncSetAttribute(k_mlp_layer<BN, SPLIT_A, SPLIT_W, HEAD, GROUPED>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)Cfg::kSmemBytes) != cudaSuccess)
            return fail(BRL_E_LAUNCH, "brl_mlp_forward: cannot reserve %u bytes of shared memory", Cfg::kSmemBytes);
        attr_set = true;
    }
    return BRL_OK;
}

template <int BN, bool SPLIT_A, bool SPLIT_W, bool HEAD, bool GROUPED = false>
static int32_t launch_layer(cudaStream_t s, const void* a_hi, const void* a_lo, int k_in, const void* w_hi, const void* w_lo,
                            int n_valid_rows, const LayerArgs& args, const PoolArgs* pool = nullptr) {
    using Cfg = LayerCfg<BN, SPLIT_A, SPLIT_W>;
    CUtensorMap ta_hi, ta_lo, tw_hi, tw_lo;
    bool ok = make_map(&ta_hi, a_hi, (uint64_t)args.M, (uint64_t)k_in, (uint64_t)k_in, kBM) &&
              make_w_map<GROUPED>(&tw_hi, w_hi, (uint64_t)n_valid_rows, (uint64_t)k_in, BN, pool);
    ta_lo = ta_hi;
    tw_lo = tw_hi;
    if (ok && SPLIT_A) ok = make_map(&ta_lo, a_lo, (uint64_t)args.M, (uint64_t)k_in, (uint64_t)k_in, kBM);
    if (ok && SPLIT_W) ok = make_w_map<GROUPED>(&tw_lo, w_lo, (uint64_t)n_valid_rows, (uint64_t)k_in, BN, pool);
    if (!ok) return fail(BRL_E_LAUNCH, "brl_mlp_forward: cuTensorMapEncodeTiled failed");
    auto kern = k_mlp_layer<BN, SPLIT_A, SPLIT_W, HEAD, GROUPED>;
    if (int32_t rc = layer_attr<BN, SPLIT_A, SPLIT_W, HEAD, GROUPED>()) return rc;
    LayerArgsT<GROUPED> la{};
    static_cast<LayerArgs&>(la) = args;
    if constexpr (GROUPED) {
        la.block_model = pool->block_model;
        la.bias_stride = pool->stride / (int64_t)sizeof(float);
        la.act = pool->act;
        la.n_rows = pool->n_rows;
    }
    la.n_tiles_n = (n_valid_rows + BN - 1) / BN;
    la.n_tiles = la.n_tiles_n * ((args.M + kBM - 1) / kBM);
    const int n_sm = sm_count();
    const unsigned grid = (unsigned)(la.n_tiles < n_sm ? la.n_tiles : n_sm);  // persistent: one CTA per SM
    kern<<<grid, kMlpThreads, Cfg::kSmemBytes, s>>>(ta_hi, ta_lo, tw_hi, tw_lo, la);
    return BRL_OK;
}

// counters of the fused forward live behind the four activation buffers of the scratch
static inline size_t fused_ready_bytes(int64_t n_envs) { return (size_t)(4 * 2 * ((n_envs + 2 * kBM - 1) / (2 * kBM))) * sizeof(uint32_t); }

// co-resident CTA pairs of the fused kernel (the dependency waits need every launched pair to be running), with its shared-memory
// attribute set on the first call per device; also called ahead of a stream capture (brl_duplicate_match).  0 = failure.
template <bool SPLIT, bool GROUPED = false>
static int fused_pairs() {
    using Cfg = FusedCfg<SPLIT>;
    auto kern = k_mlp_fused<SPLIT, GROUPED>;
    static int max_pairs_dev[kMaxDevices] = {};
    int& max_pairs = max_pairs_dev[device_slot()];
    if (max_pairs == 0) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes) != cudaSuccess) {
            fail(BRL_E_LAUNCH, "brl_mlp_forward: cannot reserve %u bytes of shared memory", Cfg::kSmemBytes);
            return 0;
        }
        const int n_sm = sm_count();
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)(n_sm & ~1));
        cfg.blockDim = dim3(kFusedThreads);
        cfg.dynamicSmemBytes = Cfg::kSmemBytes;
        cudaLaunchAttribute at{};
        at.id = cudaLaunchAttributeClusterDimension;
        at.val.clusterDim.x = 2;
        at.val.clusterDim.y = 1;
        at.val.clusterDim.z = 1;
        cfg.attrs = &at;
        cfg.numAttrs = 1;
        int n_clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&n_clusters, kern, &cfg) != cudaSuccess || n_clusters <= 0) {
            cudaGetLastError();
            n_clusters = n_sm / 2;
        }
        max_pairs = n_clusters < n_sm / 2 ? n_clusters : n_sm / 2;
    }
    return max_pairs;
}

template <bool SPLIT, bool GROUPED = false>
static int32_t launch_fused(cudaStream_t s, const void* obs, const unsigned char* blob, const MlpLayout& L, __nv_bfloat16* const buf_hi[2],
                            __nv_bfloat16* const buf_lo[2], uint32_t* ready, float* logits, float* value, int M, const ActArgs& act,
                            const PoolArgs* pool = nullptr) {
    using Cfg = FusedCfg<SPLIT>;
    FusedArgsT<GROUPED> fa{};
    bool ok = true;
    for (int l = 0; l < 5 && ok; ++l) {
        const void* a_hi = l == 0 ? obs : (const void*)buf_hi[(l - 1) & 1];
        const void* a_lo = l == 0 ? obs : (const void*)buf_lo[(l - 1) & 1];
        const uint32_t w_box = l == 4 ? kHeadPad / 2 : kFusedBN / 2;
        ok = make_map(&fa.a_hi[l], a_hi, (uint64_t)M, (uint64_t)L.k_in[l], (uint64_t)L.k_in[l], kBM) &&
             make_w_map<GROUPED>(&fa.w_hi[l], blob + L.w_hi[l], (uint64_t)L.n_out[l], (uint64_t)L.k_in[l], w_box, pool);
        fa.a_lo[l] = fa.a_hi[l];
        fa.w_lo[l] = fa.w_hi[l];
        if (ok && SPLIT && l > 0) ok = make_map(&fa.a_lo[l], a_lo, (uint64_t)M, (uint64_t)L.k_in[l], (uint64_t)L.k_in[l], kBM);
        if (ok && SPLIT) ok = make_w_map<GROUPED>(&fa.w_lo[l], blob + L.w_lo[l], (uint64_t)L.n_out[l], (uint64_t)L.k_in[l], w_box, pool);
        fa.bias[l] = reinterpret_cast<const float*>(blob + L.bias[l]);
        if (l < 4) {
            fa.out_hi[l] = buf_hi[l & 1];
            fa.out_lo[l] = SPLIT ? buf_lo[l & 1] : nullptr;
            if (ok && SPLIT)
                ok = make_map_store(&fa.st_hi[l], buf_hi[l & 1], (uint64_t)M, (uint64_t)kHidden, (uint64_t)kHidden) &&
                     make_map_store(&fa.st_lo[l], buf_lo[l & 1], (uint64_t)M, (uint64_t)kHidden, (uint64_t)kHidden);
        }
    }
    if (!ok) return fail(BRL_E_LAUNCH, "brl_mlp_forward: cuTensorMapEncodeTiled failed");
    static_assert(sizeof(fa) <= 4096, "kernel parameters");
    fa.logits = logits;
    fa.value = value;
    fa.act = act;
    fa.ready = ready;
    if constexpr (GROUPED) {
        fa.block_model = pool->block_model;
        fa.bias_stride = pool->stride / (int64_t)sizeof(float);
        fa.n_rows = pool->n_rows;
    }
    fa.M = M;
    fa.nmb = (M + 2 * kBM - 1) / (2 * kBM);
    fa.tiles_per_layer = fa.nmb * kFusedTilesN;
    fa.n_tiles = 4 * fa.tiles_per_layer + fa.nmb;
    auto kern = k_mlp_fused<SPLIT, GROUPED>;
    const int max_pairs = fused_pairs<SPLIT, GROUPED>();
    if (max_pairs == 0) return BRL_E_LAUNCH;
    if (cudaMemsetAsync(ready, 0, fused_ready_bytes(M), s) != cudaSuccess) return check_launch("brl_mlp_forward (memset)");
    const int n_pairs = fa.n_tiles < max_pairs ? fa.n_tiles : max_pairs;
    kern<<<(unsigned)(2 * n_pairs), kFusedThreads, Cfg::kSmemBytes, s>>>(fa);
    return BRL_OK;
}

__global__ void __launch_bounds__(256) k_gather_obs_rows(const uint4* __restrict__ src, const int32_t* __restrict__ index,
                                                         uint4* __restrict__ dst, int64_t n, int w) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * w) return;
    const int64_t r = i / w;
    const int c = (int)(i - r * w);
    dst[i] = src[(int64_t)index[r] * w + c];
}

// the grouped gather: launched for the grouping's capacity, it reads the padded row count from device memory and the threads
// past it exit; index -1 marks a padding row of a group, gathered as zeros
__global__ void __launch_bounds__(256) k_gather_obs_rows_grouped(const uint4* __restrict__ src, const int32_t* __restrict__ index,
                                                                 uint4* __restrict__ dst, const int32_t* __restrict__ n_rows, int w) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)*n_rows * w) return;
    const int64_t r = i / w;
    const int c = (int)(i - r * w);
    const int32_t e = index[r];
    dst[i] = e >= 0 ? src[(int64_t)e * w + c] : make_uint4(0u, 0u, 0u, 0u);
}

}  // namespace brl

using namespace brl;

extern "C" {

int64_t brl_mlp_packed_bytes(void) { return (int64_t)mlp_layout().total; }
int64_t brl_mlp_scratch_bytes(int64_t n_envs) {  // 4 activation buffers bf16[n, 1024] + the fused forward's tile counters
    return n_envs * (int64_t)kHidden * 2 * 4 + (int64_t)((fused_ready_bytes(n_envs) + 255) & ~(size_t)255);
}

int32_t brl_mlp_pack(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    for (int k = 0; k < 13; ++k)
        if (b[k] == nullptr) return fail(BRL_E_BUFFER, "brl_mlp_pack: buffer %d is NULL", k);
    BRL_REQUIRE(b[12], "packed");
    const MlpLayout L = mlp_layout();
    unsigned char* blob = static_cast<unsigned char*>(b[12]);
    for (int l = 0; l < 5; ++l) {
        const int64_t total = (int64_t)L.n_out[l] * L.k_in[l];
        const bool head = l == 4;
        k_mlp_pack<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
            static_cast<const float*>(b[l]), static_cast<const float*>(b[6 + l]),
            head ? static_cast<const float*>(b[5]) : nullptr, head ? static_cast<const float*>(b[11]) : nullptr,
            reinterpret_cast<__nv_bfloat16*>(blob + L.w_hi[l]), reinterpret_cast<__nv_bfloat16*>(blob + L.w_lo[l]),
            reinterpret_cast<float*>(blob + L.bias[l]), L.k_in[l], L.n_out[l], head ? 38 : kHidden, head ? 1 : 0);
    }
    return check_launch("brl_mlp_pack");
}

int32_t brl_obs_to_bf16(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "obs");
    BRL_REQUIRE(b[1], "obs_bf16");
    const int64_t n = p->n_envs * kObsDimM;
    const unsigned grid = (unsigned)((n / 8 + 255) / 256);
    if (p->flags & BRL_F_OBS_U8)
        k_obs_to_bf16<uint8_t><<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const uint8_t*>(b[0]), static_cast<__nv_bfloat16*>(b[1]), n);
    else
        k_obs_to_bf16<float><<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<const float*>(b[0]), static_cast<__nv_bfloat16*>(b[1]), n);
    return check_launch("brl_obs_to_bf16");
}

}  // extern "C"

// the forward's path: one persistent launch for the whole net once the batch fills the machine, per-layer launches below;
// BRL_F_TUNE_MLP_LAYERS / BRL_F_TUNE_MLP_FUSED force one of them
static bool fused_forward(const BrlParams* p) {
    if (p->flags & BRL_F_TUNE_MLP_LAYERS) return false;
    return (p->flags & BRL_F_TUNE_MLP_FUSED) != 0 || p->n_envs >= kPairMinM;
}

// forward (+ optional fused categorical) shared by brl_mlp_forward, brl_policy_act and brl_policy_act_rows.  GROUPED
// (launch_policy_grouped): `blob` is a pool of nets, row block b of the batch runs net pool->block_model[b], the kernels stop at
// the padded row count *pool->n_rows, and the head epilogue writes action / logits by env (the per-layer head included: no
// categorical launch).
template <bool GROUPED = false>
static int32_t mlp_forward_impl(const char* who, cudaStream_t s, const BrlParams* p, const void* obs, const unsigned char* blob,
                                __nv_bfloat16* scratch, float* logits, float* value, const ActArgs& act, const PoolArgs* pool = nullptr) {
    int32_t rc = BRL_OK;
    if (p->n_envs > (int64_t)1 << 30) return fail(BRL_E_OPAQUE, "%s: n_envs too large", who);
    if (encode_fn() == nullptr) return fail(BRL_E_LAUNCH, "%s: cuTensorMapEncodeTiled not available from the driver", who);
    const bool split = !(p->flags & BRL_F_MLP_BF16);
    const int M = (int)p->n_envs;
    const MlpLayout L = mlp_layout();
    const size_t act_elems = (size_t)M * kHidden;
    __nv_bfloat16* buf_hi[2] = {scratch, scratch + act_elems};
    __nv_bfloat16* buf_lo[2] = {scratch + 2 * act_elems, scratch + 3 * act_elems};
    if (fused_forward(p)) {
        uint32_t* ready = reinterpret_cast<uint32_t*>(scratch + 4 * act_elems);
        rc = split ? launch_fused<true, GROUPED>(s, obs, blob, L, buf_hi, buf_lo, ready, logits, value, M, act, pool)
                   : launch_fused<false, GROUPED>(s, obs, blob, L, buf_hi, buf_lo, ready, logits, value, M, act, pool);
        if (rc != BRL_OK) return rc;
        return check_launch(who);
    }
    // per-layer launches.  The head reads buffer 1, so buffer 0 is free to hold logits / value the caller did not ask for.
    float* lg = (logits && !act.row_index) ? logits : reinterpret_cast<float*>(buf_hi[0]);  // listed batch: compact here, scattered below
    float* vl = value ? value : reinterpret_cast<float*>(buf_lo[0]);
    const void* in_hi = obs;
    const void* in_lo = nullptr;
    for (int l = 0; l < 5; ++l) {
        LayerArgs a{};
        a.bias = reinterpret_cast<const float*>(blob + L.bias[l]);
        a.M = M;
        a.n_total = kHidden;
        a.k_blocks = (L.k_in[l] + kBK - 1) / kBK;
        const void* w_hi = blob + L.w_hi[l];
        const void* w_lo = blob + L.w_lo[l];
        if (l < 4) {
            a.out_hi = buf_hi[l & 1];
            a.out_lo = split ? buf_lo[l & 1] : nullptr;
            // 128 x 256 tiles move fewer operand bytes per MMA (the L2 -> SM fill rate, ~64 B/clk, is what bounds
            // these 1-CTA tiles): measured faster for the single-product mode; the split mode runs 128 x 128 tiles
            if (!split) rc = launch_layer<256, false, false, false, GROUPED>(s, in_hi, in_lo, L.k_in[l], w_hi, w_lo, kHidden, a, pool);
            else if (l == 0) rc = launch_layer<128, false, true, false, GROUPED>(s, in_hi, in_lo, L.k_in[l], w_hi, w_lo, kHidden, a, pool);
            else rc = launch_layer<128, true, true, false, GROUPED>(s, in_hi, in_lo, L.k_in[l], w_hi, w_lo, kHidden, a, pool);
            in_hi = a.out_hi;
            in_lo = a.out_lo;
        } else {
            a.logits = GROUPED ? logits : lg;
            a.value = GROUPED ? nullptr : vl;
            rc = split ? launch_layer<kHeadPad, true, true, true, GROUPED>(s, in_hi, in_lo, L.k_in[l], w_hi, w_lo, kHeadPad, a, pool)
                       : launch_layer<kHeadPad, false, false, true, GROUPED>(s, in_hi, in_lo, L.k_in[l], w_hi, w_lo, kHeadPad, a, pool);
        }
        if (rc != BRL_OK) return rc;
    }
    rc = check_launch(who);
    if (GROUPED || rc != BRL_OK || act.action == nullptr) return rc;
    if (act.row_index && value != nullptr) return fail(BRL_E_OPAQUE, "%s: a row-indexed batch below the fused-launch size has no value output", who);
    return launch_categorical(s, lg, act.mask, act.action, act.log_prob, M, act.sample, act.seed, act.env_offset, act.step, act.row_index,
                              act.row_index ? logits : nullptr);
}

namespace brl {

// ---- the grouped forward: brl_policy_act_grouped and the device loops of brl_duplicate_match / brl_evaluate_match -------------
// Every env listed in rows[0, *n_rows) is forwarded by the net of its kGroupRows-row block (block_model) out of the pool of
// `n_models` nets, and the head epilogue reads mask[env] and writes action[env] / logits[env] (`logits`: f32[total, 38] or NULL).
// The padded row count *n_rows (brl_model_rows' offsets[M]) is read on the device only: the gather, the launches and their tensor
// maps are sized for `capacity` rows, and the threads and row blocks past the count exit at once.  Row -1 (a group's padding)
// gathers zeros and its outputs are dropped.  The path is fused_forward's rule on `capacity` and the BRL_F_TUNE_MLP_* bits of
// `flags` (BRL_F_MLP_BF16 selects the single-product mode).
int32_t launch_policy_grouped(cudaStream_t s, int32_t flags, int64_t capacity, int n_models, const void* obs,
                              const unsigned char* pool, unsigned char* scratch, const uint8_t* mask, int32_t* action,
                              const int32_t* rows, const int32_t* block_model, const int32_t* n_rows, float* logits) {
    BrlParams p{};
    p.n_envs = capacity;
    p.flags = flags;
    uint4* gathered = reinterpret_cast<uint4*>(scratch + brl_mlp_scratch_bytes(capacity));
    const int w = kObsDimM * 2 / 16;  // uint4 per bf16 observation row
    k_gather_obs_rows_grouped<<<(unsigned)((capacity * w + 255) / 256), 256, 0, s>>>(static_cast<const uint4*>(obs), rows, gathered,
                                                                                     n_rows, w);
    ActArgs act{};
    act.mask = mask;
    act.action = action;
    act.row_index = rows;
    const PoolArgs pa{block_model, brl_mlp_pool_stride(), n_models, act, n_rows};
    return mlp_forward_impl<true>("brl_policy_act_grouped", s, &p, gathered, pool, reinterpret_cast<__nv_bfloat16*>(scratch), logits,
                                  nullptr, act, &pa);
}

// everything launch_policy_grouped sets up once per device -- the driver's tensor-map entry point, the kernels' shared-memory
// attributes, the fused kernel's co-resident pair count -- done before a stream capture begins
int32_t warm_policy_grouped(bool split) {
    if (encode_fn() == nullptr) return fail(BRL_E_LAUNCH, "device match loop: cuTensorMapEncodeTiled not available from the driver");
    int32_t rc;
    if (split) {
        if ((rc = layer_attr<128, false, true, false, true>()) || (rc = layer_attr<128, true, true, false, true>()) ||
            (rc = layer_attr<kHeadPad, true, true, true, true>()))
            return rc;
        return fused_pairs<true, true>() > 0 ? BRL_OK : BRL_E_LAUNCH;
    }
    if ((rc = layer_attr<256, false, false, false, true>()) || (rc = layer_attr<kHeadPad, false, false, true, true>()))
        return rc;
    return fused_pairs<false, true>() > 0 ? BRL_OK : BRL_E_LAUNCH;
}

}  // namespace brl

extern "C" {

int32_t brl_mlp_forward(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "obs_bf16");
    BRL_REQUIRE(b[1], "packed");
    BRL_REQUIRE(b[2], "scratch");
    BRL_REQUIRE(b[3], "logits");
    BRL_REQUIRE(b[4], "value");
    return mlp_forward_impl("brl_mlp_forward", (cudaStream_t)stream, p, b[0], static_cast<const unsigned char*>(b[1]),
                            static_cast<__nv_bfloat16*>(b[2]), static_cast<float*>(b[3]), static_cast<float*>(b[4]), ActArgs{});
}

#ifdef BRL_MLP_TRACE
int32_t brl_debug_mlp_trace(unsigned long long* out_1024x8) {
    return cudaMemcpyFromSymbol(out_1024x8, g_mlp_trace, sizeof(g_mlp_trace)) == cudaSuccess ? 0 : -1;
}
int32_t brl_debug_mlp_epi(unsigned long long* out4, int reset) {
    if (cudaMemcpyFromSymbol(out4, g_mlp_epi, sizeof(g_mlp_epi)) != cudaSuccess) return -1;
    if (reset) { unsigned long long z[4] = {0, 0, 0, 0}; cudaMemcpyToSymbol(g_mlp_epi, z, sizeof(z)); }
    return 0;
}
#endif

int64_t brl_mlp_rows_scratch_bytes(int64_t n_rows) {  // brl_mlp_scratch_bytes + the gathered bf16 observation rows
    return brl_mlp_scratch_bytes(n_rows) + n_rows * (int64_t)kObsDimM * 2;
}

// `team1_forward_pass.apply` + masked Categorical on the LISTED envs only (src/evaluation.py:124-151 without running
// either net on envs it does not decide).
int32_t brl_policy_act_rows(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "obs_bf16");
    BRL_REQUIRE(b[1], "packed");
    BRL_REQUIRE(b[2], "scratch");
    BRL_REQUIRE(b[4], "action");
    BRL_REQUIRE(b[5], "row_index");
    if (b[3] != nullptr && (reinterpret_cast<uintptr_t>(b[3]) & 1u)) return fail(BRL_E_BUFFER, "brl_policy_act_rows: mask is misaligned");
    if (b[7] != nullptr && (reinterpret_cast<uintptr_t>(b[7]) & 7u)) return fail(BRL_E_BUFFER, "brl_policy_act_rows: logits is misaligned");
    // gather the listed rows' observations (one 960-byte bf16 row per thread group) behind the forward's scratch, run the forward
    // on the compact batch, and let the head epilogue read mask[env] and write action[env] / log_prob[env] / logits[env]
    const cudaStream_t s = (cudaStream_t)stream;
    const int64_t n = p->n_envs;
    unsigned char* scratch = static_cast<unsigned char*>(b[2]);
    uint4* gathered = reinterpret_cast<uint4*>(scratch + brl_mlp_scratch_bytes(n));
    const int w = kObsDimM * 2 / 16;  // uint4 per bf16 observation row
    k_gather_obs_rows<<<(unsigned)((n * w + 255) / 256), 256, 0, s>>>(static_cast<const uint4*>(b[0]), static_cast<const int32_t*>(b[5]),
                                                                       gathered, n, w);
    ActArgs act{};
    act.mask = static_cast<const uint8_t*>(b[3]);
    act.action = static_cast<int32_t*>(b[4]);
    act.log_prob = static_cast<float*>(b[6]);
    act.seed = p->seed;
    act.env_offset = p->env_offset;
    act.step = p->step;
    act.sample = (p->flags & BRL_F_SAMPLE) ? 1 : 0;
    act.row_index = static_cast<const int32_t*>(b[5]);
    return mlp_forward_impl("brl_policy_act_rows", s, p, gathered, static_cast<const unsigned char*>(b[1]),
                            reinterpret_cast<__nv_bfloat16*>(scratch), static_cast<float*>(b[7]), nullptr, act);
}

int64_t brl_mlp_pool_stride(void) { return (int64_t)mlp_layout().total; }  // a multiple of 256: every section keeps its TMA alignment

int64_t brl_model_rows_capacity(int64_t n_envs, int64_t n_models) {  // every group rounded up to kGroupRows rows
    if (n_envs <= 0 || n_models <= 0) return 0;
    const int64_t groups = n_models < n_envs ? n_models : n_envs;
    return (n_envs + groups * (kGroupRows - 1)) / kGroupRows * kGroupRows;
}

int64_t brl_policy_grouped_scratch_bytes(int64_t n_envs, int64_t n_models) {
    return brl_mlp_rows_scratch_bytes(brl_model_rows_capacity(n_envs, n_models));
}

// `team_forward_pass.apply` + masked argmax for every listed env with ITS net out of a pool (src/evaluation.py:124-151 for all
// matches of workspace/eval_selfplay_league.py at once): the rows come grouped by net and padded per group (brl_model_rows),
// so every kGroupRows-row block runs one net; the weight operands are 3-D tensor maps over the stacked blobs.
int32_t brl_policy_act_grouped(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "obs_bf16");
    BRL_REQUIRE(b[1], "pool");
    BRL_REQUIRE(b[2], "scratch");
    BRL_REQUIRE(b[4], "action");
    BRL_REQUIRE(b[5], "rows");
    BRL_REQUIRE(b[6], "block_model");
    // n_rows is typically offsets + M of brl_model_rows: one int32, so 4-byte alignment is all it needs
    if (b[8] == nullptr) return fail(BRL_E_BUFFER, "brl_policy_act_grouped: buffer 'n_rows' is NULL");
    if (reinterpret_cast<uintptr_t>(b[8]) & 3u) return fail(BRL_E_BUFFER, "brl_policy_act_grouped: n_rows is misaligned");
    if (b[3] != nullptr && (reinterpret_cast<uintptr_t>(b[3]) & 1u)) return fail(BRL_E_BUFFER, "brl_policy_act_grouped: mask is misaligned");
    if (b[7] != nullptr && (reinterpret_cast<uintptr_t>(b[7]) & 7u)) return fail(BRL_E_BUFFER, "brl_policy_act_grouped: logits is misaligned");
    if (p->k_steps <= 0) return fail(BRL_E_OPAQUE, "brl_policy_act_grouped: k_steps (the pool's model count) must be > 0");
    if (p->n_envs % kGroupRows != 0)
        return fail(BRL_E_OPAQUE, "brl_policy_act_grouped: n_envs (padded rows) must be a multiple of %d", kGroupRows);
    if (p->flags & BRL_F_SAMPLE) return fail(BRL_E_OPAQUE, "brl_policy_act_grouped: sampling is not supported (argmax only)");
    return launch_policy_grouped((cudaStream_t)stream, p->flags, p->n_envs, p->k_steps, b[0], static_cast<const unsigned char*>(b[1]),
                                 static_cast<unsigned char*>(b[2]), static_cast<const uint8_t*>(b[3]), static_cast<int32_t*>(b[4]),
                                 static_cast<const int32_t*>(b[5]), static_cast<const int32_t*>(b[6]), static_cast<const int32_t*>(b[8]),
                                 static_cast<float*>(b[7]));
}

int32_t brl_policy_act(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "obs_bf16");
    BRL_REQUIRE(b[1], "packed");
    BRL_REQUIRE(b[2], "scratch");
    BRL_REQUIRE(b[4], "action");
    for (int k : {3, 5, 6, 7})
        if (b[k] != nullptr && (reinterpret_cast<uintptr_t>(b[k]) & (k == 3 ? 1u : 7u)) != 0)
            return fail(BRL_E_BUFFER, "brl_policy_act: buffer %d is misaligned", k);
    ActArgs act{};
    act.mask = static_cast<const uint8_t*>(b[3]);
    act.action = static_cast<int32_t*>(b[4]);
    act.log_prob = static_cast<float*>(b[5]);
    act.seed = p->seed;
    act.env_offset = p->env_offset;
    act.step = p->step;
    act.sample = (p->flags & BRL_F_SAMPLE) ? 1 : 0;
    if (p->flags & BRL_F_SEED_SALT) {
        act.seed_salt = static_cast<const uint64_t*>(b[8]);
        if (act.seed_salt == nullptr || (reinterpret_cast<uintptr_t>(b[8]) & 7u)) return fail(BRL_E_BUFFER, "brl_policy_act: BRL_F_SEED_SALT needs an 8-byte aligned buffer [8]");
        if (!fused_forward(p))
            return fail(BRL_E_OPAQUE, "brl_policy_act: BRL_F_SEED_SALT is supported by the fused launch only (n_envs >= %d, no BRL_F_TUNE_MLP_LAYERS)",
                        kPairMinM);
    }
    return mlp_forward_impl("brl_policy_act", (cudaStream_t)stream, p, b[0], static_cast<const unsigned char*>(b[1]),
                            static_cast<__nv_bfloat16*>(b[2]), static_cast<float*>(b[7]), static_cast<float*>(b[6]), act);
}

}  // extern "C"
