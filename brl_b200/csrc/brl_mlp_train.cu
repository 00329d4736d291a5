// brl_mlp_train.cu -- the PPO update's trip through the policy/value net on the 5th-gen tensor cores
// (SURVEY 8f-1): `jax.value_and_grad(_loss_fn)(params, ...)` of src/update.py:91-167 for one minibatch,
// i.e. forward of the "DeepMind" MLP (src/models.py:23-33) with the activations kept, the PPO loss head
// (brl_ppo_loss, csrc/brl_ppo.cu) and the backward GEMMs, producing d total_loss / d params as ONE flat
// fp32 buffer in the optimizer's order.  No library GEMM and no autograd tape: every product runs on
// tcgen05 with the same three-term bf16 split as the rollout forward (brl_mlp.cu), so gradients are
// fp32-class (the reference differentiates in fp32).
//
// All three GEMM shapes are  C[M, N] = A[M, K] . Bt[N, K]^T, so one pipeline (k_train_fused: TMA producer lane,
// single-lane tcgen05.mma issuer, four epilogue warps, persistent tiles, double-buffered TMEM accumulator) serves all
// of them; they differ in the epilogue and in how the operands lie in memory:
//   forward  h_l  = relu(h_{l-1} . W_l + b_l)      A = h_{l-1} [B, in] K-major     Bt^T = W_l [in, out]  MN-major
//   dgrad    dz_{l-1} = (dz_l . W_l^T) * (h_{l-1} > 0)   A = dz_l [B, out] K-major  Bt = W_l [in, out]    K-major
//   wgrad    dW_l = h_{l-1}^T . dz_l               A^T = h_{l-1} [B, in] MN-major  Bt^T = dz_l [B, out]  MN-major
// i.e. ONE copy of the weights, in haiku's own [in, out] orientation (bf16 hi / lo, "Wn"), feeds the forward (as an
// MN-major operand) and the dgrad (as a K-major one): training never transposes anything.
// The wgrad contracts over the batch, i.e. over the ROW index of the row-major activations and dz's the other
// two GEMMs read and write.  No transposed copies are made: the wgrad stages {64 features x 64 samples} TMA
// boxes of those same arrays and hands them to tcgen05.mma as MN-major operands (feature index contiguous,
// umma_desc_mn_sw128), so the same kernel serves it too.  Bias gradients are column sums of the dz's.
#include "common.h"
#include "mlp_device.cuh"
#include "ppo_gram.cuh"

namespace brl {

constexpr int kNumLayers = 5;  // four hidden layers + the fused policy/value head (38 + 1 columns, padded to 64)

// ---- flat fp32 parameter / gradient buffer: LAYERS order, w then b (brl_b200/optim.py flatten_params) ----
struct FlatLayout {
    size_t w[6], b[6], total;
};
__host__ __device__ inline FlatLayout flat_layout() {
    FlatLayout F{};
    size_t off = 0;
    for (int l = 0; l < 6; ++l) {
        const size_t in = l == 0 ? kObsDimM : kHidden, out = l < 4 ? kHidden : (l == 4 ? 38 : 1);
        F.w[l] = off; off += in * out;
        F.b[l] = off; off += out;
    }
    F.total = off;
    return F;
}

// ---- training blob: per layer (4 hidden + the fused 64-wide head) the bias in fp32 and W[in, out_pad] as bf16 hi / lo ----
struct TrainBlob {
    size_t bias[kNumLayers], wn_hi[kNumLayers], wn_lo[kNumLayers], total;
    int k_in[kNumLayers], n_pad[kNumLayers];
};
__host__ __device__ inline TrainBlob train_blob() {
    TrainBlob T{};
    size_t off = 0;
    for (int l = 0; l < kNumLayers; ++l) {
        T.k_in[l] = l == 0 ? kObsDimM : kHidden;
        T.n_pad[l] = l == 4 ? kHeadPad : kHidden;
        const size_t bytes = (size_t)T.k_in[l] * T.n_pad[l] * 2;
        T.wn_hi[l] = off; off += bytes;     // lo directly above hi: the pair is one 4-D / 3-D tensor map
        T.wn_lo[l] = off; off += bytes;
        T.bias[l] = off; off += (size_t)T.n_pad[l] * 4;
        off = (off + 255) & ~(size_t)255;
    }
    T.total = off;
    return T;
}

// row stride of a learner's flat parameters / gradients / moments in a population's [K, stride] buffers: 256-byte rows keep
// every learner's float4 accesses aligned
__host__ __device__ inline size_t param_stride() { return (flat_layout().total + 63) & ~(size_t)63; }

// ---- optimizer step + re-pack in one pass (or the pack alone) -----------------------------------------------------
// optax.chain(clip_by_global_norm, adam(eps)) over the flat buffer exactly as brl_adam_apply (csrc/brl_ppo.cu), and in the
// same pass the refreshed parameter goes out as bf16 hi / lo (weights, same [in, out] orientation) or fp32 (biases) into the
// training blob.  The four hidden layers (w and b ranges all multiples of 4 floats) take the 128-bit path; the head's
// (1024 x 38, 38, 1024 x 1, 1) ranges are remapped element-wise into its 64-wide padded tile.
struct AdamPackArgs {
    float* p;
    const float* g;
    float* m;
    float* v;
    const double* sumsq;
    unsigned char* blob;
    float max_norm, lr, b1, b2, eps, bc1, bc2;
    FlatLayout F;
    TrainBlob T;
};

template <class A>  // AdamPackArgs, or a learner's AdamLearnerView
__device__ __forceinline__ float adam_elem(const A& a, float p, float g, float& m, float& v, float scale) {
    // the roundings spelled out: which products the compiler contracts into an FMA depends on where the scalars live
    // (parameter space or registers), and every instantiation must give the bits of brl_mlp_adam_step
    const float gi = g * scale;
    m = __fmaf_rn(m, a.b1, __fmul_rn(gi, 1.0f - a.b1));
    v = __fmaf_rn(v, a.b2, __fmul_rn(gi, __fmul_rn(gi, 1.0f - a.b2)));
    return p - a.lr * (m / a.bc1) / (sqrtf(v / a.bc2) + a.eps);
}
__device__ __forceinline__ void split_pair(float v0, float v1, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = pack_bf16x2(v0 - __low2float(h), v1 - __high2float(h));
}

template <bool ADAM, class A>  // AdamPackArgs, or a learner's AdamLearnerView
__device__ __forceinline__ void adam_pack_body(const A& a) {
    float scale = 1.0f;
    if (ADAM && a.max_norm > 0.0f) {  // optax.clip_by_global_norm: g * (max_norm / norm) only when norm >= max_norm
        const float norm = (float)sqrt(*a.sumsq);
        if (!(norm < a.max_norm)) scale = a.max_norm / norm;
    }
    const size_t n_hidden = a.F.w[4];  // flat ranges [0, w[4]) = w0, b0 .. w3, b3, every boundary a multiple of 4
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i4 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i4 < n_hidden / 4; i4 += stride) {
        const size_t i = 4 * i4;
        float4 p4 = reinterpret_cast<const float4*>(a.p)[i4];
        if (ADAM) {
            const float4 g4 = reinterpret_cast<const float4*>(a.g)[i4];
            float4 m4 = reinterpret_cast<float4*>(a.m)[i4], v4 = reinterpret_cast<float4*>(a.v)[i4];
            p4.x = adam_elem(a, p4.x, g4.x, m4.x, v4.x, scale);
            p4.y = adam_elem(a, p4.y, g4.y, m4.y, v4.y, scale);
            p4.z = adam_elem(a, p4.z, g4.z, m4.z, v4.z, scale);
            p4.w = adam_elem(a, p4.w, g4.w, m4.w, v4.w, scale);
            reinterpret_cast<float4*>(a.p)[i4] = p4;
            reinterpret_cast<float4*>(a.m)[i4] = m4;
            reinterpret_cast<float4*>(a.v)[i4] = v4;
        }
        int l = 0;
#pragma unroll
        for (int k = 1; k < 4; ++k)
            if (i >= a.F.w[k]) l = k;
        if (i < a.F.b[l]) {  // weight: same offset inside Wn[l] (n_pad == n_out for the hidden layers)
            const size_t e = i - a.F.w[l];
            uint2 hi, lo;
            split_pair(p4.x, p4.y, hi.x, lo.x);
            split_pair(p4.z, p4.w, hi.y, lo.y);
            *reinterpret_cast<uint2*>(a.blob + a.T.wn_hi[l] + 2 * e) = hi;
            *reinterpret_cast<uint2*>(a.blob + a.T.wn_lo[l] + 2 * e) = lo;
        } else {
            *reinterpret_cast<float4*>(a.blob + a.T.bias[l] + 4 * (i - a.F.b[l])) = p4;
        }
    }
    // head: w4 [1024, 38], b4 [38], w5 [1024, 1], b5 [1] -> Wn[4] [1024, 64] (columns 39..63 stay zero), bias[4] [64]
    for (size_t i = n_hidden + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.F.total; i += stride) {
        float p = a.p[i];
        if (ADAM) {
            float m = a.m[i], v = a.v[i];
            p = adam_elem(a, p, a.g[i], m, v, scale);
            a.p[i] = p;
            a.m[i] = m;
            a.v[i] = v;
        }
        size_t e;        // element of Wn[4], or
        int bias_col = -1;
        if (i < a.F.b[4]) { const size_t r = i - a.F.w[4]; e = (r / 38) * kHeadPad + r % 38; }
        else if (i < a.F.w[5]) { bias_col = (int)(i - a.F.b[4]); e = 0; }
        else if (i < a.F.b[5]) { e = (i - a.F.w[5]) * kHeadPad + 38; }
        else { bias_col = 38; e = 0; }
        if (bias_col >= 0) {
            reinterpret_cast<float*>(a.blob + a.T.bias[4])[bias_col] = p;
        } else {
            const __nv_bfloat16 h = __float2bfloat16_rn(p);
            reinterpret_cast<__nv_bfloat16*>(a.blob + a.T.wn_hi[4])[e] = h;
            reinterpret_cast<__nv_bfloat16*>(a.blob + a.T.wn_lo[4])[e] = __float2bfloat16_rn(p - __bfloat162float(h));
        }
    }
}
template <bool ADAM>
__global__ void __launch_bounds__(256) k_adam_pack(const __grid_constant__ AdamPackArgs a) {
    pdl_trigger();
    pdl_wait();
    adam_pack_body<ADAM, AdamPackArgs>(a);
}

// the optimizer steps of K learners (brl_mlp_adam_step_grouped), blockIdx.y = learner: learner k's params / grads / m / v
// lie k * param_stride() floats after learner 0's, its blob k * T.total bytes, its |g|^2 k * sumsq_stride doubles
struct AdamLearner {
    float max_norm, lr, b1, b2, eps, bc1, bc2;
};
struct GroupedAdamArgs {
    AdamPackArgs a;  // learner 0's buffers
    long long sumsq_stride;
    AdamLearner l[BRL_MAX_LEARNERS];
};
// learner k's view of GroupedAdamArgs: its own pointers and scalars; the layouts stay in the parameter space (a local copy of
// their arrays, indexed at run time, would live in local memory)
struct AdamLearnerView {
    float* p;
    const float* g;
    float* m;
    float* v;
    const double* sumsq;
    unsigned char* blob;
    float max_norm, lr, b1, b2, eps, bc1, bc2;
    const FlatLayout& F;
    const TrainBlob& T;
};
__global__ void __launch_bounds__(256) k_adam_pack_grouped(const __grid_constant__ GroupedAdamArgs g) {
    pdl_trigger();
    pdl_wait();
    const int k = blockIdx.y;
    const size_t n = param_stride() * k;
    const AdamLearner& l = g.l[k];
    const AdamLearnerView a{g.a.p + n, g.a.g + n, g.a.m + n, g.a.v + n, g.a.sumsq + k * g.sumsq_stride, g.a.blob + k * g.a.T.total,
                            l.max_norm, l.lr, l.b1, l.b2, l.eps, l.bc1, l.bc2, g.a.F, g.a.T};
    adam_pack_body<true, AdamLearnerView>(a);
}

// ---- per-minibatch scratch -------------------------------------------------------------------------------
constexpr int kMaxOps = 9;  // GEMMs of one fused launch (forward: 5, backward: 9)
constexpr int kTraceTiles = 4096;
// tile counters of the two fused launches: per launch, per op: one counter per 128-row block of the op's OUTPUT (batch
// rows for forward / dgrad, input features for wgrad) + one total
__host__ __device__ inline int ready_blocks(int64_t B) {
    const int nb = (int)((B + kBM - 1) / kBM);
    return nb > kHidden / kBM ? nb : kHidden / kBM;
}
__host__ __device__ inline size_t ready_words(int64_t B) { return (size_t)2 * kMaxOps * (size_t)(ready_blocks(B) + 1); }
struct TrainScratch {
    size_t obs;                                   // bf16 [B, 480]
    size_t h_hi[4], h_lo[4];                      // activations of layers 1..4, bf16 hi / lo [B, 1024]
    size_t dz_hi[4], dz_lo[4];                    // d loss / d pre-activation of layers 1..4, bf16 hi / lo [B, 1024]
    size_t dz5_hi, dz5_lo;                        // head: [B, 64] (38 logits, value, zero padding)
    size_t logits, value, dlogits, dvalue;        // f32 [B, 38], [B]
    size_t ready;                                 // u32 tile counters of the fused launches (ready_words)
    size_t trace;                                 // u64 [2][kTraceTiles][8] %globaltimer stamps (tune bit 3, scripts/exp_train_trace.py)
    size_t total;
};
__host__ inline TrainScratch train_scratch(int64_t B) {
    TrainScratch S{};
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~(size_t)255; return o; };
    S.obs = take((size_t)B * kObsDimM * 2);
    for (int l = 0; l < 4; ++l) {
        S.h_hi[l] = take((size_t)B * kHidden * 2);
        S.h_lo[l] = take((size_t)B * kHidden * 2);
        S.dz_hi[l] = take((size_t)B * kHidden * 2);
        S.dz_lo[l] = take((size_t)B * kHidden * 2);
    }
    S.dz5_hi = take((size_t)B * kHeadPad * 2);
    S.dz5_lo = take((size_t)B * kHeadPad * 2);
    S.logits = take((size_t)B * 38 * 4);
    S.value = take((size_t)B * 4);
    S.dlogits = take((size_t)B * 38 * 4);
    S.dvalue = take((size_t)B * 4);
    S.ready = take(ready_words(B) * sizeof(uint32_t));
    S.trace = take((size_t)2 * kTraceTiles * 8 * sizeof(unsigned long long));
    S.total = off;
    return S;
}

// ---- minibatch gather of the observation: obs[index[b]] (f32 / u8 0-1, or bf16) -> bf16 [B, 480] -------------------
template <class T>
__device__ __forceinline__ uint16_t obs_bits(T v) { return (float)v != 0.0f ? (uint16_t)0x3F80u : (uint16_t)0u; }
template <>
__device__ __forceinline__ uint16_t obs_bits<__nv_bfloat16>(__nv_bfloat16 v) { return *reinterpret_cast<uint16_t*>(&v); }

template <class T>
__device__ __forceinline__ void gather_obs_body(const T* __restrict__ obs, const int32_t* __restrict__ index, int64_t B,
                                                uint16_t* __restrict__ out) {
    // 8 consecutive observation bits per thread: one 128-bit store
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * (kObsDimM / 8)) return;
    const int64_t b = i / (kObsDimM / 8);
    const int c = (int)(i % (kObsDimM / 8)) * 8;
    const T* src = obs + (index ? (int64_t)index[b] : b) * kObsDimM + c;
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) w[k] = (uint32_t)obs_bits<T>(src[2 * k]) | ((uint32_t)obs_bits<T>(src[2 * k + 1]) << 16);
    *reinterpret_cast<uint4*>(out + b * kObsDimM + c) = make_uint4(w[0], w[1], w[2], w[3]);
}
template <class T>
__global__ void __launch_bounds__(256) k_gather_obs(const T* __restrict__ obs, const int32_t* __restrict__ index, int64_t B,
                                                    uint16_t* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    gather_obs_body<T>(obs, index, B, out);
}
// K learners (blockIdx.y): learner k's observation and index from row k of the trajectory table, its rows to out + k * stride
template <class T>
__global__ void __launch_bounds__(256) k_gather_obs_grouped(const long long* __restrict__ traj, int64_t B, uint16_t* out,
                                                            long long out_stride) {
    pdl_trigger();
    pdl_wait();
    const long long* t = traj + 8 * blockIdx.y;
    gather_obs_body<T>(reinterpret_cast<const T*>(t[0]), reinterpret_cast<const int32_t*>(t[1]), B,
                       reinterpret_cast<uint16_t*>(reinterpret_cast<char*>(out) + blockIdx.y * out_stride));
}

// bias gradients: db[c] = sum_b dz[b, c].  Hidden layers: column sums of dz (hi + lo); a block owns 64 columns of one
// layer, thread = (row group of 32, column pair), then a shared-memory reduction over the row groups.  Last block: the
// head, column sums of the fp32 d loss / d (logits, value) themselves.
struct BiasArgs {
    const __nv_bfloat16* hi[4];
    const __nv_bfloat16* lo[4];
    const float* dlogits;  // [B, 38]
    const float* dvalue;   // [B]
    float* grads;
    double* sumsq;         // += sum of squares of the bias gradients, or NULL
    int64_t B;
    FlatLayout F;
    GramArgs gram;         // deferred spectral-norm statistic: its serial tail runs in one spare block (n_gram partials; 0 = none)
    int n_gram;
};
template <class A>  // BiasArgs, or a learner's BiasLearnerView
__device__ __forceinline__ void bias_sumsq(const A& a, float v) {  // called by whole warps
    if (a.sumsq == nullptr) return;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(a.sumsq, (double)v);
}
template <class A>  // BiasArgs, or a learner's BiasLearnerView
__device__ __forceinline__ void bias_grad_body(const A& a) {
    // a block either sums bias columns (red) or runs the Gram tail (GramSmem): one shared buffer for both
    constexpr size_t kSmemBytes = sizeof(GramSmem) > sizeof(float) * 32 * 65 ? sizeof(GramSmem) : sizeof(float) * 32 * 65;
    __shared__ __align__(16) unsigned char smem_raw[kSmemBytes];
    float (*red)[65] = reinterpret_cast<float (*)[65]>(smem_raw);
    const int tid = threadIdx.x, rg = tid >> 5, cp = tid & 31;  // 32 row groups x 32 column pairs
    const int blocks_per_layer = kHidden / 64;
    if ((int)blockIdx.x > 4 * blocks_per_layer) {
        // one spare block (the bias sums occupy 65 of the 148 SMs): sum + eigen-solve of the illegal-probability Gram matrix
        // for the logged illegal_action_loss (ppo_gram.cuh), deferred to here when its coefficient is 0 so that the serial
        // tail runs beside the bias sums instead of between the loss head and the backward GEMMs
        gram_tail(a.gram, a.n_gram, *reinterpret_cast<GramSmem*>(smem_raw));
        return;
    }
    if ((int)blockIdx.x < 4 * blocks_per_layer) {
        const int l = blockIdx.x / blocks_per_layer, c0 = (blockIdx.x % blocks_per_layer) * 64;
        const __nv_bfloat162* hi = reinterpret_cast<const __nv_bfloat162*>(a.hi[l] + c0) + cp;
        const __nv_bfloat162* lo = reinterpret_cast<const __nv_bfloat162*>(a.lo[l] + c0) + cp;
        float s0 = 0.0f, s1 = 0.0f;
#pragma unroll 4
        for (int64_t b = rg; b < a.B; b += 32) {
            const float2 h = __bfloat1622float2(hi[b * (kHidden / 2)]), r = __bfloat1622float2(lo[b * (kHidden / 2)]);
            s0 += h.x + r.x;
            s1 += h.y + r.y;
        }
        red[rg][2 * cp] = s0;
        red[rg][2 * cp + 1] = s1;
        __syncthreads();
        if (tid < 64) {
            float s = 0.0f;
#pragma unroll
            for (int k = 0; k < 32; ++k) s += red[k][tid];
            a.grads[a.F.b[l] + c0 + tid] = s;
            bias_sumsq(a, s * s);
        }
    } else {  // head: thread = (row group of 16, column), 39 columns
        const int c = tid & 63, g16 = tid >> 6;
        float s = 0.0f;
        if (c < kHeadValid)
            for (int64_t b = g16; b < a.B; b += 16) s += c < 38 ? a.dlogits[b * 38 + c] : a.dvalue[b];
        red[g16][c] = s;
        __syncthreads();
        if (tid < 64) {  // both warps whole: bias_sumsq shuffles
            float tot = 0.0f;
            if (tid < kHeadValid) {
#pragma unroll
                for (int k = 0; k < 16; ++k) tot += red[k][tid];
                if (tid < 38) a.grads[a.F.b[4] + tid] = tot;
                else a.grads[a.F.b[5]] = tot;
            }
            bias_sumsq(a, tot * tot);
        }
    }
}
__global__ void __launch_bounds__(1024) k_bias_grad(const __grid_constant__ BiasArgs a) {
    pdl_trigger();
    pdl_wait();
    bias_grad_body<BiasArgs>(a);
}
// K learners (blockIdx.y), every learner's grid with the spare block; `a` holds learner 0's buffers.  The spare block runs
// learner k's deferred Gram tail when its illegal_l2_coef is 0 and the statistic is asked for.
struct GroupedBiasArgs {
    BiasArgs a;
    const long long* traj;   // [K][8] trajectory table (index, mask of the Gram tail)
    const float* coefs;      // [K][4] loss coefficients (illegal_l2_coef: column 3)
    const float* logits;     // learner 0's forward logits
    float* stats;            // [K][8]
    unsigned char* acc;      // [K][BRL_PPO_SCRATCH_BYTES]
    long long sc_stride;     // bytes
    int illegal_stat, n_gram;
};
// learner k's view of GroupedBiasArgs (as AdamLearnerView: the layout and the dz pointers stay in the parameter space)
struct ShiftedRows {  // learner 0's per-layer pointers, read as learner k's
    const __nv_bfloat16* const* base;
    long long off;
    __device__ __forceinline__ const __nv_bfloat16* operator[](int l) const {
        return reinterpret_cast<const __nv_bfloat16*>(reinterpret_cast<const char*>(base[l]) + off);
    }
};
struct BiasLearnerView {
    ShiftedRows hi, lo;
    const float* dlogits;
    const float* dvalue;
    float* grads;
    double* sumsq;
    int64_t B;
    const FlatLayout& F;
    GramArgs gram;
    int n_gram;
};
__global__ void __launch_bounds__(1024) k_bias_grad_grouped(const __grid_constant__ GroupedBiasArgs g) {
    pdl_trigger();
    pdl_wait();
    const int k = blockIdx.y;
    const long long off = k * g.sc_stride;
    auto sc = [&](auto* p) { return (decltype(p))((const char*)p + off); };
    unsigned char* acc = g.acc + (size_t)k * BRL_PPO_SCRATCH_BYTES;
    GramArgs gram{};
    int n_gram = 0;
    if ((int)blockIdx.x > 4 * (kHidden / 64)) {
        if (!g.illegal_stat || g.coefs[4 * k + 3] != 0.0f) return;
        const long long* t = g.traj + 8 * k;
        gram = gram_args_at(sc(g.logits), reinterpret_cast<const int32_t*>(t[1]), reinterpret_cast<const uint8_t*>(t[2]), g.a.B, acc,
                            g.stats + 8 * k + 6);
        n_gram = g.n_gram;
    }
    const BiasLearnerView a{{g.a.hi, off}, {g.a.lo, off}, sc(g.a.dlogits), sc(g.a.dvalue), g.a.grads + k * param_stride(),
                            reinterpret_cast<double*>(acc) + 14, g.a.B, g.a.F, gram, n_gram};
    bias_grad_body<BiasLearnerView>(a);
}

// ---- the GEMM ---------------------------------------------------------------------------------------------
enum { kEpiFwd = 0, kEpiHead = 1, kEpiDgrad = 2, kEpiWgrad = 3 };

struct GemmArgs {
    int M, k_blocks, n_tiles_n, n_tiles;
    // kEpiFwd / kEpiDgrad: bf16 hi / lo outputs [M, ld_out]
    const float* bias;                 // kEpiFwd, kEpiHead
    __nv_bfloat16 *out_hi, *out_lo;
    int ld_out;
    const __nv_bfloat16* relu_src;     // kEpiDgrad: the forward activation (hi part) this gradient flows through, [M, ld_out]
    // kEpiWgrad: fp32 output [M, ld_c], columns < n_c; column n_c (the value head of the fused head tile) -> c2[row]
    float* c;
    float* c2;
    int ld_c, n_c;
    double* sumsq;                     // kEpiWgrad: += sum of squares of the gradient block (for clip_by_global_norm), or NULL
    // kEpiHead
    float *logits, *value;
};

constexpr uint32_t kMnBox = 64 * kBK * 2;  // one {64 features, 64 samples} box of an MN-major operand: 8 KB

template <bool MN>
__device__ __forceinline__ uint64_t operand_desc(uint32_t saddr) {
    return MN ? umma_desc_mn_sw128(saddr, kMnBox) : umma_desc_sw128(saddr);
}

// 32 accumulator columns of this thread's row; t_off2 != 0 (k_train_fused): the tile's products live in two column
// blocks t_off2 apart (x.w_hi terms | x_hi.w_lo term) and their sum is the result
__device__ __forceinline__ void tmem_ld32_sum(uint32_t taddr, uint32_t t_off2, uint32_t (&r)[32]) {
    tmem_ld32(taddr, r);
    if (t_off2 != 0u) {
        uint32_t r2[32];
        tmem_ld32(taddr + t_off2, r2);
#pragma unroll
        for (int k = 0; k < 32; ++k) r[k] = __float_as_uint(__uint_as_float(r[k]) + __uint_as_float(r2[k]));
    }
}

// forward / dgrad rows: x -> bf16 hi / lo, 128-bit stores
template <int EPI>
__device__ __forceinline__ void epilogue_act_row(uint32_t t_row, int n_cols, int n0, int row, bool row_ok, const GemmArgs& a, uint32_t t_off2) {
#pragma unroll 1
    for (int c0 = 0; c0 < n_cols; c0 += 32) {
        uint32_t r[32];
        tmem_ld32_sum(t_row + (uint32_t)c0, t_off2, r);
        if (!row_ok) continue;
        const size_t ro = (size_t)row * a.ld_out + n0 + c0;
        uint32_t keep[16];
        if (EPI == kEpiDgrad) {
            const uint4* ps = reinterpret_cast<const uint4*>(a.relu_src + ro);
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const uint4 m = ps[v];
                keep[4 * v] = m.x; keep[4 * v + 1] = m.y; keep[4 * v + 2] = m.z; keep[4 * v + 3] = m.w;
            }
        }
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) {
            float x0 = __uint_as_float(r[2 * jj]), x1 = __uint_as_float(r[2 * jj + 1]);
            if (EPI == kEpiFwd) {
                const float2 bb = __ldg(reinterpret_cast<const float2*>(a.bias + n0 + c0) + jj);  // warp-uniform
                x0 = fmaxf(x0 + bb.x, 0.0f);
                x1 = fmaxf(x1 + bb.y, 0.0f);
            } else {  // relu'(h) = [h > 0]; h >= 0 always, so "non-zero" is "positive"
                if ((keep[jj] & 0x00007FFFu) == 0u) x0 = 0.0f;
                if ((keep[jj] & 0x7FFF0000u) == 0u) x1 = 0.0f;
            }
            __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
            hi[jj] = *reinterpret_cast<uint32_t*>(&h);
            lo[jj] = pack_bf16x2(x0 - __low2float(h), x1 - __high2float(h));
        }
        uint4* ph = reinterpret_cast<uint4*>(a.out_hi + ro);
        uint4* pl = reinterpret_cast<uint4*>(a.out_lo + ro);
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            ph[v] = make_uint4(hi[4 * v], hi[4 * v + 1], hi[4 * v + 2], hi[4 * v + 3]);
            pl[v] = make_uint4(lo[4 * v], lo[4 * v + 1], lo[4 * v + 2], lo[4 * v + 3]);
        }
    }
}

// head rows (epilogue_head_row of the rollout forward, over the two column blocks): columns 0..37 logits, 38 value
__device__ __forceinline__ void epilogue_head_row2(uint32_t t_row, uint32_t t_off2, const float* __restrict__ bias, bool row_ok,
                                                   float* __restrict__ logits_row, float* __restrict__ value_row) {
    uint32_t r0[32], r1[32];
    tmem_ld32_sum(t_row, t_off2, r0);
    tmem_ld32_sum(t_row + 32u, t_off2, r1);
    if (row_ok) {
        float2* pl = reinterpret_cast<float2*>(logits_row);
#pragma unroll
        for (int jj = 0; jj < 16; ++jj)
            pl[jj] = make_float2(__uint_as_float(r0[2 * jj]) + __ldg(bias + 2 * jj), __uint_as_float(r0[2 * jj + 1]) + __ldg(bias + 2 * jj + 1));
#pragma unroll
        for (int jj = 0; jj < 3; ++jj)
            pl[16 + jj] = make_float2(__uint_as_float(r1[2 * jj]) + __ldg(bias + 32 + 2 * jj),
                                      __uint_as_float(r1[2 * jj + 1]) + __ldg(bias + 32 + 2 * jj + 1));
        *value_row = __uint_as_float(r1[6]) + __ldg(bias + 38);
    }
}

// wgrad rows: the accumulator IS the gradient block; thread = one input feature (row of W)
template <int BN>
__device__ __forceinline__ void epilogue_wgrad_row(uint32_t t_row, int n0, int row, bool row_ok, const GemmArgs& a, uint32_t t_off2) {
    float ss = 0.0f;  // this row's share of |g|^2 (padding columns of the head tile are exact zeros)
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t r[32];
        tmem_ld32_sum(t_row + (uint32_t)c0, t_off2, r);
        if (!row_ok) continue;
#pragma unroll
        for (int j = 0; j < 32; ++j) ss = fmaf(__uint_as_float(r[j]), __uint_as_float(r[j]), ss);
        if (a.c2 != nullptr) {  // fused head tile: 38 policy columns (row pitch 38 floats: 8-byte aligned) + the value column
#pragma unroll
            for (int j = 0; j < 32; j += 2) {
                const int col = n0 + c0 + j;
                if (col + 1 < a.n_c)
                    *reinterpret_cast<float2*>(a.c + (size_t)row * a.ld_c + col) = make_float2(__uint_as_float(r[j]), __uint_as_float(r[j + 1]));
                else if (col == a.n_c)
                    a.c2[row] = __uint_as_float(r[j]);
            }
        } else {
            float4* pc = reinterpret_cast<float4*>(a.c + (size_t)row * a.ld_c + n0 + c0);
#pragma unroll
            for (int v = 0; v < 8; ++v)
                pc[v] = make_float4(__uint_as_float(r[4 * v]), __uint_as_float(r[4 * v + 1]), __uint_as_float(r[4 * v + 2]),
                                    __uint_as_float(r[4 * v + 3]));
        }
    }
    if (a.sumsq != nullptr) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if ((threadIdx.x & 31) == 0) atomicAdd(a.sumsq, (double)ss);
    }
}

// ---- all GEMMs of the forward (or of the backward) as ONE persistent launch ----------------------------------------
// At a 1024-sample minibatch each GEMM is ~128 tiles of ~6 us on 148 SMs: run one launch per GEMM and the fixed costs
// (launch gap, barrier / tensor-memory set-up, pipeline fill, the un-overlapped epilogue of each CTA's single tile)
// are as large as the main loops.  Here the tiles of up to kMaxOps GEMMs form one list walked round-robin by one CTA
// per SM, with the same producer / MMA / epilogue pipeline as k_gemm_tc running straight across op boundaries.
// Dependencies: a forward / dgrad tile reads only rows [m0, m0 + 128) of its producer's output, so it waits for that
// 128-row block (producer's n-tiles x 4 epilogue warps arrivals); a wgrad tile contracts over the whole batch and
// waits for the producer's total.  Epilogue warps publish with st.global + __threadfence + atomicAdd; the TMA producer
// acquires the counter and crosses into the async proxy before the tile's first load.  Tiles depend only on tiles
// earlier in the list, every CTA takes its tiles in list order and the grid never exceeds the SM count (1 CTA / SM),
// so the waits cannot deadlock; spins are bounded (a protocol bug traps instead of hanging the GPU).
struct FusedOp {
    // One bulk-tensor request per operand per stage: a (hi, lo) pair is ONE map with a trailing dimension of 2 whose stride
    // is the distance between the two arrays -- K-major {64 k, rows, 2}, MN-major {64 features, 64 samples, 64-feature
    // chunks, 2} -- so the box lands as [hi tile][lo tile], the layout the MMA descriptors expect.  (Measured: a stage costs
    // ~0.14 us per REQUEST whatever its size, scripts/exp_train_trace.py.)  The unsplit 0/1 observation keeps 2-D maps.
    CUtensorMap a, w;
    GemmArgs g;
    int epi, split_a;
    int a_mn, w_mn;          // operand stored with its M / N index contiguous (MN-major) instead of K
    int tile0;               // index of this op's first tile in the list
    int dep;                 // producing op of this launch, -1 = none (inputs complete before the launch)
    int dep_all;             // 1: wait for all of the producer's tiles, 0: for its row block m0 / 128
    uint32_t dep_count;      // arrivals that complete the awaited counter
};
struct FusedTrainArgs {
    FusedOp op[kMaxOps];
    int n_ops, n_tiles, nmb;
    uint32_t* ready;         // [n_ops][nmb + 1]: per-row-block counters, then the op's total
    unsigned long long* trace;  // NULL, or [n_tiles][8] time stamps: dep wait begin / end, loads issued, first MMA, last MMA issued, accumulator seen, published
};
// The same launch for K learners (brl_ppo_grad_grouped).  Every op's tensor maps carry a trailing learner coordinate, and
// its pointers are learner 0's: learner k's scratch, blob, gradient and |g|^2 lie k strides further.  Op o's tile range
// holds the K learners' tiles of that op back to back (op.g.n_tiles is ONE learner's count), so a learner's chain waits
// are filled by the other learners' tiles of the same op.  Counters: ready[(o * K + k) * (nmb + 1) + row block].
struct GroupedTrainArgs {
    FusedTrainArgs f;
    int K;
    long long sc_stride, blob_stride;  // bytes
    long long grad_stride;             // floats
    long long sumsq_stride;            // doubles
};
template <bool GROUPED>
using TrainArgsT = std::conditional_t<GROUPED, GroupedTrainArgs, FusedTrainArgs>;
__device__ __forceinline__ const FusedTrainArgs& fused_of(const FusedTrainArgs& a) { return a; }
__device__ __forceinline__ const FusedTrainArgs& fused_of(const GroupedTrainArgs& a) { return a.f; }

// learner k's epilogue arguments: every output pointer moved by its buffer's stride
__device__ __forceinline__ GemmArgs learner_gemm(const GroupedTrainArgs& a, const GemmArgs& g, int k) {
    GemmArgs r = g;
    auto sc = [&](auto* p) { return p ? (decltype(p))((const char*)p + k * a.sc_stride) : p; };
    r.out_hi = sc(g.out_hi);
    r.out_lo = sc(g.out_lo);
    r.relu_src = sc(g.relu_src);
    r.logits = sc(g.logits);
    r.value = sc(g.value);
    r.bias = g.bias ? reinterpret_cast<const float*>(reinterpret_cast<const char*>(g.bias) + k * a.blob_stride) : nullptr;
    r.c = g.c ? g.c + k * a.grad_stride : nullptr;
    r.c2 = g.c2 ? g.c2 + k * a.grad_stride : nullptr;
    r.sumsq = g.sumsq ? g.sumsq + k * a.sumsq_stride : nullptr;
    return r;
}

// FBN = tile width of the fused launches: 64 keeps the most tiles in flight, 128 moves a third fewer operand bytes from
// L2 per FLOP (the measured bound at minibatch sizes) and relies on tiles of different ops to fill the SMs.
template <int kFBN>
struct FusedTrainCfg {
    static constexpr uint32_t kABytes = kBM * kBK * 2, kWBytes = kFBN * kBK * 2;
    static constexpr uint32_t kStageBytes = 2 * kABytes + 2 * kWBytes;  // A_hi, A_lo (unused when the A operand is exact), W_hi, W_lo
    static constexpr int kStages = (int)(kSmemBudget / kStageBytes);
    static constexpr uint32_t kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/;
};

__device__ __forceinline__ void trace_stamp(const FusedTrainArgs& a, int tile, int slot) {
    if (a.trace != nullptr && tile < kTraceTiles) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        a.trace[(size_t)tile * 8 + slot] = t;
    }
}

__device__ __forceinline__ int fused_find_op(const FusedTrainArgs& a, int tile) {
    int o = 0;
#pragma unroll 1
    for (int k = 1; k < a.n_ops; ++k)
        if (tile >= a.op[k].tile0) o = k;
    return o;
}

template <int kFBN, bool GROUPED>
__global__ void __launch_bounds__(kMlpThreads, 1) k_train_fused(const __grid_constant__ TrainArgsT<GROUPED> ga) {
    const FusedTrainArgs& a = fused_of(ga);
    using Cfg = FusedTrainCfg<kFBN>;
    constexpr int S = Cfg::kStages;
    // The main loop is bound by the shared-memory port (TMA writes + the operand reads of the SS-mode MMAs, DESIGN.md), so
    // the W_hi and W_lo tiles -- adjacent in a stage -- are consumed as ONE operand of N = 2 x kFBN: x_hi is read once for
    // both of its products, which land in two column blocks of the accumulator (x.w_hi terms | x_hi.w_lo) that the
    // epilogue adds.
    constexpr uint32_t kBufCols = 2 * kFBN, kTmemCols = 2 * kBufCols;
    extern __shared__ unsigned char smem_dyn[];
    const uint32_t base = (smem_addr(smem_dyn) + 1023u) & ~1023u;
    const uint32_t bar_base = base + S * Cfg::kStageBytes;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (S + s); };
    auto tmem_full_bar = [&](int b) { return bar_base + 8u * (2 * S + b); };
    auto tmem_empty_bar = [&](int b) { return bar_base + 8u * (2 * S + 2 + b); };
    __shared__ uint32_t tmem_base_s;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_tiles = a.n_tiles;

    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (warp == 0 && lane == 0) {
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
    asm volatile("griddepcontrol.wait;" ::: "memory");

    if (warp == 0) {
        if (lane == 0) {  // ===== TMA producer =====
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const int o = fused_find_op(a, tile);
                const FusedOp& op = a.op[o];
                int r = tile - op.tile0, k = 0;
                if constexpr (GROUPED) { k = r / op.g.n_tiles; r -= k * op.g.n_tiles; }
                const int mb = r / op.g.n_tiles_n, m0 = mb * kBM, n0 = (r % op.g.n_tiles_n) * kFBN;
                const bool split_a = op.split_a != 0, a_mn = op.a_mn != 0, w_mn = op.w_mn != 0;
                const uint32_t tx = Cfg::kABytes * (split_a ? 2u : 1u) + 2u * Cfg::kWBytes;
                trace_stamp(a, tile, 0);
                if (op.dep >= 0) {
                    size_t counter = (size_t)op.dep;
                    if constexpr (GROUPED) counter = counter * ga.K + k;
                    const uint32_t* flag = a.ready + counter * (a.nmb + 1) + (op.dep_all ? a.nmb : mb);
                    uint32_t v = 0;
                    for (uint32_t spin = 0;; ++spin) {
                        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
                        if (v >= op.dep_count) break;
                        if (spin > (1u << 24)) __trap();
                        __nanosleep(64);
                    }
                    asm volatile("fence.proxy.async;" ::: "memory");  // generic-proxy writes -> async-proxy (TMA) reads
                }
                trace_stamp(a, tile, 1);
                for (int kb = 0; kb < op.g.k_blocks; ++kb, ++it) {
                    const int s = (int)(it % S);
                    mbar_wait(empty_bar(s), ((it / S) & 1u) ^ 1u);
                    mbar_expect_tx(full_bar(s), tx);
                    const uint32_t sa = base + s * Cfg::kStageBytes;
                    const uint32_t sw = sa + 2 * Cfg::kABytes;
                    // K-major operand: {64 k, rows (, hi / lo)}; MN-major: {64 features, 64 k rows, 64-feature chunks, hi / lo}
                    if constexpr (!GROUPED) {
                        if (!a_mn) {
                            if (split_a) tma_load_3d(sa, &op.a, full_bar(s), kb * kBK, m0, 0);
                            else tma_load_2d(sa, &op.a, full_bar(s), kb * kBK, m0);
                        } else if (split_a) {
                            tma_load_4d(sa, &op.a, full_bar(s), 0, kb * kBK, m0 / 64, 0);
                        } else {
#pragma unroll
                            for (int j = 0; j < kBM / 64; ++j) tma_load_2d(sa + j * kMnBox, &op.a, full_bar(s), m0 + 64 * j, kb * kBK);
                        }
                        if (!w_mn) tma_load_3d(sw, &op.w, full_bar(s), kb * kBK, n0, 0);
                        else tma_load_4d(sw, &op.w, full_bar(s), 0, kb * kBK, n0 / 64, 0);
                    } else {  // the same boxes, one more (learner) coordinate
                        if (!a_mn) {
                            if (split_a) tma_load_4d(sa, &op.a, full_bar(s), kb * kBK, m0, 0, k);
                            else tma_load_3d(sa, &op.a, full_bar(s), kb * kBK, m0, k);
                        } else if (split_a) {
                            tma_load_5d(sa, &op.a, full_bar(s), 0, kb * kBK, m0 / 64, 0, k);
                        } else {
#pragma unroll
                            for (int j = 0; j < kBM / 64; ++j) tma_load_3d(sa + j * kMnBox, &op.a, full_bar(s), m0 + 64 * j, kb * kBK, k);
                        }
                        if (!w_mn) tma_load_4d(sw, &op.w, full_bar(s), kb * kBK, n0, 0, k);
                        else tma_load_5d(sw, &op.w, full_bar(s), 0, kb * kBK, n0 / 64, 0, k);
                    }
                }
                trace_stamp(a, tile, 2);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {  // ===== MMA issuer =====
            uint32_t it = 0, j = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++j) {
                const FusedOp& op = a.op[fused_find_op(a, tile)];
                const bool split_a = op.split_a != 0, a_mn = op.a_mn != 0, w_mn = op.w_mn != 0;
                const uint32_t majors = (a_mn ? 1u << 15 : 0u) | (w_mn ? 1u << 16 : 0u);
                const uint32_t idesc = umma_idesc_bf16(kBM, kFBN) | majors, idesc2 = umma_idesc_bf16(kBM, 2 * kFBN) | majors;
                const int k_blocks = op.g.k_blocks;
                const uint32_t buf = j & 1u;
                mbar_wait(tmem_empty_bar(buf), ((j >> 1) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t acc = tmem_acc + buf * kBufCols;
                for (int kb = 0; kb < k_blocks; ++kb, ++it) {
                    const int s = (int)(it % S);
                    mbar_wait(full_bar(s), (it / S) & 1u);
                    tc_fence_after();
                    if (kb == 0) trace_stamp(a, tile, 3);
                    const uint32_t sa_hi = base + s * Cfg::kStageBytes;
                    const uint32_t sa_lo = sa_hi + Cfg::kABytes;
                    const uint32_t sw_hi = sa_hi + 2 * Cfg::kABytes;
#pragma unroll
                    for (int k = 0; k < kBK / kUmmaK; ++k) {
                        // 16 K elements further: 32 bytes along a K-major row, 16 rows of 128 bytes in an MN-major tile
                        const uint32_t koff_a = (uint32_t)k * kUmmaK * (a_mn ? 128u : 2u), koff_w = (uint32_t)k * kUmmaK * (w_mn ? 128u : 2u);
                        const uint64_t da_hi = a_mn ? operand_desc<true>(sa_hi + koff_a) : operand_desc<false>(sa_hi + koff_a);
                        const uint64_t dw_hi = w_mn ? operand_desc<true>(sw_hi + koff_w) : operand_desc<false>(sw_hi + koff_w);
                        umma_bf16(acc, da_hi, dw_hi, idesc2, (kb | k) != 0);  // x_hi . [w_hi ; w_lo]: the W_lo tile follows W_hi
                        if (split_a) umma_bf16(acc, a_mn ? operand_desc<true>(sa_lo + koff_a) : operand_desc<false>(sa_lo + koff_a), dw_hi, idesc, 1u);
                    }
                    umma_commit(empty_bar(s));
                }
                umma_commit(tmem_full_bar(buf));
                trace_stamp(a, tile, 4);
            }
        }
    } else {  // ===== epilogue: warps 2..5, TMEM lane quarter = warp % 4 =====
        const int q = warp & 3;
        uint32_t j = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++j) {
            const int o = fused_find_op(a, tile);
            const FusedOp& op = a.op[o];
            int r = tile - op.tile0, k = 0;
            if constexpr (GROUPED) { k = r / op.g.n_tiles; r -= k * op.g.n_tiles; }
            const int mb = r / op.g.n_tiles_n, m0 = mb * kBM, n0 = (r % op.g.n_tiles_n) * kFBN;
            const uint32_t buf = j & 1u;
            mbar_wait(tmem_full_bar(buf), (j >> 1) & 1u);
            tc_fence_after();
            if (q == 0 && lane == 0) trace_stamp(a, tile, 5);
            const int row = m0 + q * 32 + lane;
            const uint32_t t_row = tmem_acc + buf * kBufCols + ((uint32_t)(q * 32) << 16);
            const bool row_ok = row < op.g.M;
            auto epilogue = [&](const GemmArgs& g) {
                if (op.epi == kEpiFwd) epilogue_act_row<kEpiFwd>(t_row, kFBN, n0, row, row_ok, g, (uint32_t)kFBN);
                else if (op.epi == kEpiDgrad) epilogue_act_row<kEpiDgrad>(t_row, kFBN, n0, row, row_ok, g, (uint32_t)kFBN);
                else if (op.epi == kEpiWgrad) epilogue_wgrad_row<kFBN>(t_row, n0, row, row_ok, g, (uint32_t)kFBN);
                else epilogue_head_row2(t_row, (uint32_t)kFBN, g.bias + n0, row_ok, g.logits + (size_t)row * 38, g.value + row);
            };
            if constexpr (GROUPED) epilogue(learner_gemm(ga, op.g, k));
            else epilogue(op.g);
            tc_fence_before();
            __syncwarp();  // orders the other lanes' stores before lane 0's fence (the grid-barrier idiom: sync, one fence, one atomic)
            if (lane == 0) {
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tmem_empty_bar(buf)) : "memory");
                __threadfence();  // cumulative: the warp's output rows are visible GPU-wide before the counts below
                size_t counter = (size_t)o;
                if constexpr (GROUPED) counter = counter * ga.K + k;
                uint32_t* cnt = a.ready + counter * (a.nmb + 1);
                atomicAdd(cnt + mb, 1u);
                atomicAdd(cnt + a.nmb, 1u);
                if (q == 0) trace_stamp(a, tile, 6);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_acc, kTmemCols);
}

// one GEMM of the update, C[m_rows, n_rows] = A . Bt^T over k_cols, as the host describes it.  A K-major operand is the
// row-major [m_rows (n_rows), k_cols] array, an MN-major one (a_mn / w_mn) the row-major [k_cols, m_rows (n_rows)] array;
// lda / ldb = row pitch in elements, *_lo = NULL for an operand that is exact in bf16 (the 0/1 observation).
struct OpSpec {
    const void *a_hi, *a_lo;
    int m_rows, lda, a_mn;
    const void *w_hi, *w_lo;
    int n_rows, ldb, w_mn, k_cols;
    int epi;
    GemmArgs g;
    int dep, dep_all;
    long long a_stride, w_stride;  // grouped launch: bytes from learner k's operand to learner k + 1's
};

// the K learners of a grouped launch and the strides between their buffers
struct GroupSpec {
    int K;
    long long sc_stride, blob_stride, grad_stride, sumsq_stride;
};

template <int kFBN, bool GROUPED = false>
static int32_t launch_fused_ops(cudaStream_t s, const OpSpec* ops, int n_ops, int nmb, uint32_t* ready, unsigned long long* trace,
                                const char* what, const GroupSpec* grp = nullptr) {
    using Cfg = FusedTrainCfg<kFBN>;
    TrainArgsT<GROUPED> ga{};
    FusedTrainArgs* fa_ptr;
    if constexpr (GROUPED) fa_ptr = &ga.f;
    else fa_ptr = &ga;
    FusedTrainArgs& fa = *fa_ptr;
    const int K = GROUPED ? grp->K : 1;
    int tiles = 0;
    for (int i = 0; i < n_ops; ++i) {
        const OpSpec& o = ops[i];
        FusedOp& f = fa.op[i];
        // a grouped map has one more dimension, the learner, `stride` bytes apart
        auto map_nd = [&](CUtensorMap* m, const void* ptr, int rank, uint64_t* dims, uint64_t* str, uint32_t* box, long long stride) {
            if (GROUPED) {
                dims[rank] = (uint64_t)K;
                str[rank - 1] = (uint64_t)stride;
                box[rank] = 1;
                ++rank;
            }
            return make_map_nd(m, ptr, rank, dims, str, box);
        };
        // (hi, lo) pair of one operand as a single map; feat = the operand's M / N extent, pitch in elements
        auto pair_map = [&](CUtensorMap* m, const void* hi, const void* lo, bool mn, int feat, int pitch, uint32_t box_feat, long long stride) {
            if (static_cast<const char*>(lo) <= static_cast<const char*>(hi)) return false;  // the trailing dimension steps hi -> lo
            const uint64_t gap = (uint64_t)(static_cast<const char*>(lo) - static_cast<const char*>(hi));
            if (!mn) {  // K-major: [feat, k_cols]
                uint64_t dims[5] = {(uint64_t)o.k_cols, (uint64_t)feat, 2}, str[4] = {(uint64_t)pitch * 2, gap};
                uint32_t box[5] = {(uint32_t)kBK, box_feat, 2};
                return map_nd(m, hi, 3, dims, str, box, stride);
            }
            // MN-major: [k_cols, feat], features in chunks of 64
            uint64_t dims[5] = {64, (uint64_t)o.k_cols, (uint64_t)((feat + 63) / 64), 2}, str[4] = {(uint64_t)pitch * 2, 128, gap};
            uint32_t box[5] = {64, (uint32_t)kBK, box_feat / 64, 2};
            return map_nd(m, hi, 4, dims, str, box, stride);
        };
        bool ok = pair_map(&f.w, o.w_hi, o.w_lo, o.w_mn != 0, o.n_rows, o.ldb, kFBN, o.w_stride);
        if (ok && o.a_lo) {
            ok = pair_map(&f.a, o.a_hi, o.a_lo, o.a_mn != 0, o.m_rows, o.lda, kBM, o.a_stride);
        } else if (ok && !GROUPED) {
            ok = o.a_mn ? make_map(&f.a, o.a_hi, (uint64_t)o.k_cols, (uint64_t)o.m_rows, (uint64_t)o.lda, 64)
                        : make_map(&f.a, o.a_hi, (uint64_t)o.m_rows, (uint64_t)o.k_cols, (uint64_t)o.lda, kBM);
        } else if (ok) {  // make_map's boxes plus the learner dimension
            const uint64_t rows = o.a_mn ? (uint64_t)o.k_cols : (uint64_t)o.m_rows, cols = o.a_mn ? (uint64_t)o.m_rows : (uint64_t)o.k_cols;
            uint64_t dims[5] = {cols, rows}, str[4] = {(uint64_t)o.lda * 2};
            uint32_t box[5] = {(uint32_t)kBK, o.a_mn ? 64u : (uint32_t)kBM};
            ok = map_nd(&f.a, o.a_hi, 2, dims, str, box, o.a_stride);
        }
        if (!ok) return fail(BRL_E_LAUNCH, "%s: cuTensorMapEncodeTiled failed", what);
        f.g = o.g;
        f.g.M = o.m_rows;
        f.g.k_blocks = (o.k_cols + kBK - 1) / kBK;
        f.g.n_tiles_n = (o.n_rows + kFBN - 1) / kFBN;
        f.g.n_tiles = f.g.n_tiles_n * ((o.m_rows + kBM - 1) / kBM);
        f.epi = o.epi;
        f.split_a = o.a_lo != nullptr;
        f.a_mn = o.a_mn;
        f.w_mn = o.w_mn;
        f.tile0 = tiles;
        tiles += K * f.g.n_tiles;
        f.dep = o.dep;
        f.dep_all = o.dep_all;
        if (o.dep >= 0) f.dep_count = 4u * (uint32_t)(o.dep_all ? fa.op[o.dep].g.n_tiles : fa.op[o.dep].g.n_tiles_n);
    }
    fa.n_ops = n_ops;
    fa.n_tiles = tiles;
    fa.nmb = nmb;
    fa.ready = ready;
    fa.trace = trace;
    if constexpr (GROUPED) {
        ga.K = K;
        ga.sc_stride = grp->sc_stride;
        ga.blob_stride = grp->blob_stride;
        ga.grad_stride = grp->grad_stride;
        ga.sumsq_stride = grp->sumsq_stride;
    }
    static bool attr_set_dev[kMaxDevices] = {};
    bool& attr_set = attr_set_dev[device_slot()];
    if (!attr_set) {
        if (cudaFuncSetAttribute(k_train_fused<kFBN, GROUPED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::kSmemBytes) != cudaSuccess)
            return fail(BRL_E_LAUNCH, "%s: cannot reserve %u bytes of shared memory", what, Cfg::kSmemBytes);
        attr_set = true;
    }
    const int n_sm = sm_count();
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(tiles < n_sm ? tiles : n_sm));  // one CTA per SM: all of them co-resident
    cfg.blockDim = dim3(kMlpThreads);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cfg.stream = s;
    cudaLaunchAttribute at{};
    at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &at;
    cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, k_train_fused<kFBN, GROUPED>, ga) != cudaSuccess) return check_launch(what);
    return BRL_OK;
}

}  // namespace brl

using namespace brl;

static int train_ops(OpSpec* fwd, OpSpec* bwd, unsigned char* sc, const unsigned char* blob, float* grads, double* grad_sumsq, int B);

// one learner's BrlAdamParams -> the optimizer scalars of AdamPackArgs / AdamLearner (learner < 0: a solo step)
template <class D>
static int32_t adam_scalars(const char* what, long long learner, const BrlAdamParams& p, D& d) {
    if (p.n != (int64_t)flat_layout().total || p.step <= 0) {
        char at[32] = "";
        if (learner >= 0) snprintf(at, sizeof(at), "learner %lld: ", learner);
        return fail(BRL_E_OPAQUE, "%s: %sn must be brl_mlp_num_params() and step (1-based) > 0", what, at);
    }
    d.max_norm = p.max_grad_norm; d.lr = p.lr; d.b1 = p.beta1; d.b2 = p.beta2; d.eps = p.eps;
    d.bc1 = 1.0f - powf(p.beta1, (float)p.step);
    d.bc2 = 1.0f - powf(p.beta2, (float)p.step);
    return BRL_OK;
}

extern "C" {

int64_t brl_mlp_num_params(void) { return (int64_t)flat_layout().total; }
int64_t brl_mlp_train_blob_bytes(void) { return (int64_t)train_blob().total; }
int64_t brl_mlp_param_stride(void) { return (int64_t)param_stride(); }
int64_t brl_mlp_train_scratch_bytes(int64_t batch) { return batch > 0 ? (int64_t)train_scratch(batch).total : 0; }
int64_t brl_mlp_train_trace_offset(int64_t batch) { return batch > 0 ? (int64_t)train_scratch(batch).trace : 0; }

static unsigned adam_pack_grid() {
    const size_t items = flat_layout().w[4] / 4;  // the 128-bit body; the head's 40 K elements ride along
    size_t g = (items + 255) / 256;
    return (unsigned)(g > 148 * 8 ? 148 * 8 : g);
}

int32_t brl_mlp_pack_train(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    BRL_REQUIRE(b[0], "params");
    BRL_REQUIRE(b[1], "blob");
    cudaStream_t s = (cudaStream_t)stream;
    AdamPackArgs a{};
    a.p = static_cast<float*>(b[0]);
    a.blob = static_cast<unsigned char*>(b[1]);
    a.F = flat_layout();
    a.T = train_blob();
    // the head tile's padding columns (39..63) and bias entries are never written by the packer: zero them once here
    if (cudaMemsetAsync(a.blob + a.T.wn_hi[4], 0, a.T.total - a.T.wn_hi[4], s) != cudaSuccess) return check_launch("brl_mlp_pack_train");
    launch_pdl(k_adam_pack<false>, dim3(adam_pack_grid()), dim3(256), 0, s, a);
    return check_launch("brl_mlp_pack_train");
}

int32_t brl_mlp_adam_step(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    if (opaque == nullptr || len != sizeof(BrlAdamParams))
        return fail(BRL_E_OPAQUE, "brl_mlp_adam_step: opaque must be one BrlAdamParams (%zu bytes), got %zu", sizeof(BrlAdamParams), len);
    static const char* names[] = {"params", "grads", "m", "v", "sumsq", "blob"};
    AdamPackArgs a{};
    int32_t rc = check_buffers("brl_mlp_adam_step", b, names, 6, 0, 0x3Fu & ~(1u << 4));
    if (rc != BRL_OK || (rc = adam_scalars("brl_mlp_adam_step", -1, *static_cast<const BrlAdamParams*>(opaque), a)) != BRL_OK) return rc;
    a.p = static_cast<float*>(b[0]);
    a.g = static_cast<const float*>(b[1]);
    a.m = static_cast<float*>(b[2]);
    a.v = static_cast<float*>(b[3]);
    a.sumsq = static_cast<const double*>(b[4]);
    a.blob = static_cast<unsigned char*>(b[5]);
    a.F = flat_layout();
    a.T = train_blob();
    launch_pdl(k_adam_pack<true>, dim3(adam_pack_grid()), dim3(256), 0, (cudaStream_t)stream, a);
    return check_launch("brl_mlp_adam_step");
}

// brl_ppo_grad, and with `anchored` brl_ppo_grad_anchored: buffers [13] anchor logits, [14] kl_coef add the KL term
static int32_t ppo_grad_impl(const char* what, bool anchored, brl_stream_t stream, void** b, const void* opaque, size_t len) {
    if (opaque == nullptr || len != sizeof(BrlPpoParams))
        return fail(BRL_E_OPAQUE, "%s: opaque must be one BrlPpoParams (%zu bytes), got %zu", what, sizeof(BrlPpoParams), len);
    const BrlPpoParams* p = static_cast<const BrlPpoParams*>(opaque);
    if (anchored && p->batch == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL
    if (p->batch <= 0 || p->batch > (1 << 24)) return fail(BRL_E_OPAQUE, "%s: batch must be in [1, 2^24]", what);
    static const char* names[] = {"obs", "blob", "scratch", "index", "mask", "action", "old_log_prob", "old_value", "advantages",
                                  "targets", "grads", "stats", "acc", "anchor_logits", "kl_coef"};
    const int32_t rc = check_buffers(what, b, names, anchored ? 15 : 13, 1u << 3, 1u << 0 | 1u << 1 | 1u << 2 | 1u << 10);
    if (rc != BRL_OK) return rc;
    if (encode_fn() == nullptr) return fail(BRL_E_LAUNCH, "%s: cuTensorMapEncodeTiled not available from the driver", what);
    cudaStream_t s = (cudaStream_t)stream;
    // 3. loss head + its backward (src/update.py:97-162)
    struct PpoHead {
        void** b;
        BrlPpoParams params;
        bool defer_illegal;
        PpoAnchor anchor;
    };
    // only the logged statistic needs the spectral norm: off the critical path
    PpoHead head{b, *p, p->illegal_l2_coef == 0.0f, PpoAnchor{}};
    if (anchored) head.anchor = PpoAnchor{static_cast<const float*>(b[13]), nullptr, static_cast<const float*>(b[14])};
    head.params.flags &= (BRL_PPO_VALUE_CLIPPING | BRL_PPO_REWARD_SCALING | BRL_PPO_UNMASKED_POLICY | BRL_PPO_ILLEGAL_STAT);
    head.params.reserved = 0;
    const bool skip_illegal = head.defer_illegal && !(p->flags & BRL_PPO_ILLEGAL_STAT);  // statistic not asked for: stats[6] = NaN
    auto ppo_head = [](cudaStream_t st, const TrainHeadIO& io, const void* ctx) -> int32_t {
        const PpoHead& h = *static_cast<const PpoHead*>(ctx);
        void* loss_buffers[13] = {const_cast<float*>(io.logits), const_cast<float*>(io.value), h.b[3], h.b[4], h.b[5], h.b[6], h.b[7],
                                  h.b[8], h.b[9], io.dlogits, io.dvalue, h.b[11], h.b[12]};
        return launch_ppo_loss(st, loss_buffers, &h.params, io.dz_hi, io.dz_lo, /*acc_zeroed=*/true, h.defer_illegal,
                               h.anchor.coef ? &h.anchor : nullptr);
    };
    TrainMinibatch t{};
    t.obs = b[0];
    t.obs_flags = p->flags & (BRL_PPO_OBS_U8 | BRL_PPO_OBS_BF16);
    t.index = static_cast<const int32_t*>(b[3]);
    t.batch = p->batch;
    t.blob = static_cast<const unsigned char*>(b[1]);
    t.scratch = static_cast<unsigned char*>(b[2]);
    t.grads = static_cast<float*>(b[10]);
    t.grad_sumsq = static_cast<double*>(b[12]) + 14;  // |grads|^2 accumulates in acc[14] (input of brl_adam_apply)
    t.zero = b[12];
    t.zero_bytes = 16 * sizeof(double);
    t.tune = p->reserved;
    // deferred illegal-action statistic: its Gram tail runs in a spare block of the bias sums (gram_args reads only the
    // logits / index / mask / scratch slots of the loss buffers)
    GramArgs gram{};
    if (head.defer_illegal && !skip_illegal) {
        const TrainScratch S = train_scratch(p->batch);
        void* loss_buffers[13] = {t.scratch + S.logits, nullptr, b[3], b[4], nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, b[11], b[12]};
        gram = gram_args(loss_buffers, &head.params, static_cast<float*>(b[11]) + 6);
        t.gram = &gram;
        t.n_gram = gram_blocks(p->batch, 1024);
    }
    t.what = what;
    t.loss_head = ppo_head;
    t.ctx = &head;
    return launch_train_minibatch(s, t);
}

int32_t brl_ppo_grad(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return ppo_grad_impl("brl_ppo_grad", false, stream, b, opaque, len);
}

int32_t brl_ppo_grad_anchored(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return ppo_grad_impl("brl_ppo_grad_anchored", true, stream, b, opaque, len);
}

// ---- K learners, one optimizer step each, in the launches of one -------------------------------------------------------
// scratch: K per-learner minibatch scratches (train_scratch(B), learner k's at k * total), then the grouped launches' tile
// counters: [2 launches][kMaxOps][K][nmb + 1]
static size_t grouped_ready_offset(int64_t K, int64_t B) { return (size_t)K * train_scratch(B).total; }

int64_t brl_ppo_grad_grouped_scratch_bytes(int64_t n_learners, int64_t batch) {
    if (n_learners <= 0 || batch <= 0 || n_learners > BRL_MAX_LEARNERS || batch > (1 << 24)) return 0;
    return (int64_t)(grouped_ready_offset(n_learners, batch) + n_learners * ready_words(batch) * sizeof(uint32_t));
}

// brl_ppo_grad_grouped, and with `anchored` brl_ppo_grad_grouped_anchored: buffers [7] anchor logits table, [8] kl_coef[K]
static int32_t ppo_grad_grouped_impl(const char* what, bool anchored, brl_stream_t stream, void** b, const void* opaque, size_t len) {
    if (opaque == nullptr || len != sizeof(BrlPpoGroupedParams))
        return fail(BRL_E_OPAQUE, "%s: opaque must be one BrlPpoGroupedParams (%zu bytes), got %zu", what, sizeof(BrlPpoGroupedParams),
                    len);
    const BrlPpoGroupedParams* p = static_cast<const BrlPpoGroupedParams*>(opaque);
    if (p->n_learners < 0 || p->n_learners > BRL_MAX_LEARNERS)
        return fail(BRL_E_OPAQUE, "%s: n_learners must be in [0, %d]", what, BRL_MAX_LEARNERS);
    if (p->batch < 0 || p->batch > (1 << 24)) return fail(BRL_E_OPAQUE, "%s: batch must be in [0, 2^24]", what);
    if (p->n_learners == 0 || p->batch == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL
    static const char* names[] = {"traj", "coefs", "blob", "scratch", "grads", "stats", "acc", "anchor_logits", "kl_coef"};
    const int32_t rc = check_buffers(what, b, names, anchored ? 9 : 7, 0, 1u << 0 | 1u << 2 | 1u << 3 | 1u << 4 | 1u << 6);
    if (rc != BRL_OK) return rc;
    if (encode_fn() == nullptr) return fail(BRL_E_LAUNCH, "%s: cuTensorMapEncodeTiled not available from the driver", what);
    PpoAnchor anchor{nullptr, static_cast<const long long*>(anchored ? b[7] : nullptr), static_cast<const float*>(anchored ? b[8] : nullptr)};
    PpoGroupIO io{};  // the loss heads' arguments but the forward outputs, which launch_train_minibatch hands to the head
    io.traj = static_cast<const long long*>(b[0]);
    io.coefs = static_cast<const float*>(b[1]);
    io.sc_stride = (long long)train_scratch(p->batch).total;
    io.stats = static_cast<float*>(b[5]);
    io.acc = static_cast<unsigned char*>(b[6]);
    io.batch = p->batch;
    io.K = p->n_learners;
    io.flags = p->flags & (BRL_PPO_VALUE_CLIPPING | BRL_PPO_REWARD_SCALING | BRL_PPO_UNMASKED_POLICY | BRL_PPO_ILLEGAL_STAT);
    io.anchor = anchored ? &anchor : nullptr;
    auto ppo_heads = [](cudaStream_t st, const TrainHeadIO& head, const void* ctx) -> int32_t {
        PpoGroupIO io = *static_cast<const PpoGroupIO*>(ctx);
        io.head = head;
        return launch_ppo_loss_grouped(st, io);
    };
    const TrainGroup group{p->n_learners, io.traj, io.coefs, io.stats, (p->flags & BRL_PPO_ILLEGAL_STAT) != 0};
    TrainMinibatch t{};
    t.obs_flags = p->flags & (BRL_PPO_OBS_U8 | BRL_PPO_OBS_BF16);
    t.batch = p->batch;
    t.blob = static_cast<const unsigned char*>(b[2]);
    t.scratch = static_cast<unsigned char*>(b[3]);
    t.grads = static_cast<float*>(b[4]);
    t.grad_sumsq = static_cast<double*>(b[6]) + 14;  // learner k's |grads|^2: f64 14 of its accumulator slice
    t.zero = b[6];
    t.zero_bytes = 16 * sizeof(double);
    t.tune = p->reserved & ~8;  // the tile trace (tune bit 3) records one learner's launches
    t.what = what;
    t.loss_head = ppo_heads;
    t.ctx = &io;
    t.group = &group;
    return launch_train_minibatch((cudaStream_t)stream, t);
}

int32_t brl_ppo_grad_grouped(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return ppo_grad_grouped_impl("brl_ppo_grad_grouped", false, stream, b, opaque, len);
}

int32_t brl_ppo_grad_grouped_anchored(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return ppo_grad_grouped_impl("brl_ppo_grad_grouped_anchored", true, stream, b, opaque, len);
}

int32_t brl_mlp_adam_step_grouped(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    if ((opaque == nullptr && len != 0) || len % sizeof(BrlAdamParams) != 0)
        return fail(BRL_E_OPAQUE, "brl_mlp_adam_step_grouped: opaque must be an array of BrlAdamParams (%zu bytes each), got %zu bytes",
                    sizeof(BrlAdamParams), len);
    const int64_t K = (int64_t)(len / sizeof(BrlAdamParams));
    if (K == 0) return BRL_OK;  // no learners: a no-op, its buffers may be NULL
    if (K > BRL_MAX_LEARNERS) return fail(BRL_E_OPAQUE, "brl_mlp_adam_step_grouped: at most %d learners", BRL_MAX_LEARNERS);
    static const char* names[] = {"params", "grads", "m", "v", "acc", "blob"};
    int32_t rc = check_buffers("brl_mlp_adam_step_grouped", b, names, 6, 0, 0x3Fu);
    if (rc != BRL_OK) return rc;
    const BrlAdamParams* p = static_cast<const BrlAdamParams*>(opaque);
    GroupedAdamArgs g{};
    for (int64_t k = 0; k < K; ++k)
        if ((rc = adam_scalars("brl_mlp_adam_step_grouped", (long long)k, p[k], g.l[k])) != BRL_OK) return rc;
    g.a.p = static_cast<float*>(b[0]);
    g.a.g = static_cast<const float*>(b[1]);
    g.a.m = static_cast<float*>(b[2]);
    g.a.v = static_cast<float*>(b[3]);
    g.a.sumsq = static_cast<const double*>(b[4]) + 14;
    g.a.blob = static_cast<unsigned char*>(b[5]);
    g.a.F = flat_layout();
    g.a.T = train_blob();
    g.sumsq_stride = BRL_PPO_SCRATCH_BYTES / (long long)sizeof(double);
    launch_pdl(k_adam_pack_grouped, dim3(adam_pack_grid(), (unsigned)K), dim3(256), 0, (cudaStream_t)stream, g);
    return check_launch("brl_mlp_adam_step_grouped");
}

}  // extern "C"

// The GEMMs of one minibatch: fwd[5] and bwd[] (returns the number of backward ops)
static int train_ops(OpSpec* fwd, OpSpec* bwd, unsigned char* sc, const unsigned char* blob, float* grads, double* grad_sumsq, int B) {
    const TrainBlob T = train_blob();
    const FlatLayout F = flat_layout();
    const TrainScratch S = train_scratch(B);
    auto bf = [&](size_t off) { return reinterpret_cast<__nv_bfloat16*>(sc + off); };
    // 2. the GEMMs.  Forward: layers 1..4 (activations kept, row-major bf16 hi / lo: next layer's A, the ReLU mask, the
    //    wgrad's MN-major A) + the head.  Backward: dgrad into layer l's pre-activation, dz_l = (dz_{l+1} . W_{l+1}^T) * [h_l > 0]
    //    (S.dz_*[l-1], l = 1..4), and the wgrads dW_l = h_{l-1}^T . dz_l straight from the row-major h and dz.
    // |grads|^2 accumulates in grad_sumsq (cleared by the caller before the loss head, which runs before every wgrad)
    for (int l = 0; l < 5; ++l) {  // forward: A = previous activation (K-major), W = Wn[l] [in, out_pad] (MN-major)
        OpSpec& o = fwd[l];
        o = OpSpec{};
        o.a_hi = l == 0 ? sc + S.obs : sc + S.h_hi[l - 1];
        o.a_lo = l == 0 ? nullptr : sc + S.h_lo[l - 1];
        o.m_rows = B; o.lda = T.k_in[l];
        o.w_hi = blob + T.wn_hi[l]; o.w_lo = blob + T.wn_lo[l]; o.w_mn = 1;
        o.n_rows = T.n_pad[l]; o.ldb = T.n_pad[l]; o.k_cols = T.k_in[l];
        o.g.bias = reinterpret_cast<const float*>(blob + T.bias[l]);
        if (l < 4) {
            o.epi = kEpiFwd;
            o.g.out_hi = bf(S.h_hi[l]); o.g.out_lo = bf(S.h_lo[l]);
            o.g.ld_out = kHidden;
        } else {
            o.epi = kEpiHead;
            o.g.logits = reinterpret_cast<float*>(sc + S.logits);
            o.g.value = reinterpret_cast<float*>(sc + S.value);
        }
        o.dep = l - 1; o.dep_all = 0;
    }
    int nb = 0;
    int dgrad_op[5] = {-1, -1, -1, -1, -1};  // op index (in bwd) that produced dz of layer l (1..4)
    auto add_head_wgrad = [&] {  // [1024, 39] = h4^T . dz5 -> w4 grads (38 columns) + w5 grads (the value column)
        OpSpec& o = bwd[nb++];
        o = OpSpec{};
        o.a_hi = sc + S.h_hi[3]; o.a_lo = sc + S.h_lo[3]; o.m_rows = kHidden; o.lda = kHidden; o.a_mn = 1;
        o.w_hi = sc + S.dz5_hi; o.w_lo = sc + S.dz5_lo; o.n_rows = kHeadPad; o.ldb = kHeadPad; o.w_mn = 1; o.k_cols = B;
        o.epi = kEpiWgrad;
        o.g.c = grads + F.w[4]; o.g.ld_c = 38; o.g.n_c = 38; o.g.c2 = grads + F.w[5]; o.g.sumsq = grad_sumsq;
        o.dep = -1;
    };
    auto add_dgrad = [&](int l) {  // dz_{l+1} -> dz_l (the layer-to-layer chain of the backward)
        OpSpec& o = bwd[nb];
        o = OpSpec{};
        const int k_out = l == 4 ? kHeadPad : kHidden;  // width of dz_{l+1}
        o.a_hi = l == 4 ? sc + S.dz5_hi : sc + S.dz_hi[l];
        o.a_lo = l == 4 ? sc + S.dz5_lo : sc + S.dz_lo[l];
        o.m_rows = B; o.lda = k_out;
        o.w_hi = blob + T.wn_hi[l]; o.w_lo = blob + T.wn_lo[l]; o.n_rows = kHidden; o.ldb = k_out; o.k_cols = k_out;
        o.epi = kEpiDgrad;
        o.g.out_hi = bf(S.dz_hi[l - 1]); o.g.out_lo = bf(S.dz_lo[l - 1]);
        o.g.ld_out = kHidden;
        o.g.relu_src = bf(S.h_hi[l - 1]);
        o.dep = l == 4 ? -1 : dgrad_op[l + 1]; o.dep_all = 0;
        dgrad_op[l] = nb++;
    };
    auto add_wgrad = [&](int l) {  // wgrad of layer l (0-based parameter index l - 1): dW = h_{l-1}^T . dz_l
        OpSpec& o = bwd[nb++];
        o = OpSpec{};
        o.a_hi = l == 1 ? sc + S.obs : sc + S.h_hi[l - 2];
        o.a_lo = l == 1 ? nullptr : sc + S.h_lo[l - 2];
        o.m_rows = l == 1 ? kObsDimM : kHidden; o.lda = o.m_rows; o.a_mn = 1;
        o.w_hi = sc + S.dz_hi[l - 1]; o.w_lo = sc + S.dz_lo[l - 1]; o.n_rows = kHidden; o.ldb = kHidden; o.w_mn = 1; o.k_cols = B;
        o.epi = kEpiWgrad;
        o.g.c = grads + F.w[l - 1]; o.g.ld_c = kHidden; o.g.n_c = kHidden; o.g.sumsq = grad_sumsq;
        o.dep = dgrad_op[l]; o.dep_all = 1;
    };
    {
        // The dgrad chain dz5 -> dz4 -> ... -> dz1 is the critical path; the weight gradients only have to come after the dz they
        // contract.  Tiles are dealt round-robin in list order, so the chain goes first and every wgrad one layer behind it: no
        // CTA holds a chain tile behind a full-K wgrad tile that could have run later (0.1695 -> 0.1688 ms per step against
        // "head wgrad first, then dgrad_l / wgrad_l per layer": the chain's own latency, not queueing, is what bounds it).
        add_dgrad(4);
        add_dgrad(3);
        add_head_wgrad();
        add_wgrad(4);
        add_dgrad(2);
        add_wgrad(3);
        add_dgrad(1);
        add_wgrad(2);
        add_wgrad(1);
    }
    // a grouped launch: learner k's operands lie k scratches (activations, dz) or blobs (weights) after learner 0's
    for (OpSpec* o = fwd; o != fwd + 5; ++o) { o->a_stride = (long long)S.total; o->w_stride = (long long)T.total; }
    for (int i = 0; i < nb; ++i) {
        bwd[i].a_stride = (long long)S.total;
        bwd[i].w_stride = bwd[i].epi == kEpiWgrad ? (long long)S.total : (long long)T.total;
    }
    return nb;
}

// one fused launch of the GEMMs at the tile width `wide` selects, for one learner (grp = NULL) or a group
static int32_t launch_gemms(bool wide, cudaStream_t s, const OpSpec* ops, int n_ops, int nmb, uint32_t* ready,
                            unsigned long long* trace, const char* what, const GroupSpec* grp) {
    if (grp) return wide ? launch_fused_ops<128, true>(s, ops, n_ops, nmb, ready, trace, what, grp)
                         : launch_fused_ops<64, true>(s, ops, n_ops, nmb, ready, trace, what, grp);
    return wide ? launch_fused_ops<128>(s, ops, n_ops, nmb, ready, trace, what) : launch_fused_ops<64>(s, ops, n_ops, nmb, ready, trace, what);
}

int32_t brl::launch_train_minibatch(cudaStream_t s, const TrainMinibatch& t) {
    const TrainGroup* grp = t.group;
    const int B = (int)t.batch, K = grp ? grp->K : 1;
    const FlatLayout F = flat_layout();
    const TrainScratch S = train_scratch(B);
    unsigned char* sc = t.scratch;
    float* grads = t.grads;
    auto bf = [&](size_t off) { return reinterpret_cast<__nv_bfloat16*>(sc + off); };
    const int nmb = ready_blocks(B);
    uint32_t* ready = reinterpret_cast<uint32_t*>(sc + (grp ? grouped_ready_offset(K, B) : S.ready));
    int32_t rc = BRL_OK;

    // 0. counters and accumulators first, so that nothing but kernels (launched with programmatic dependent launch) follows
    if (cudaMemsetAsync(ready, 0, K * ready_words(B) * sizeof(uint32_t), s) != cudaSuccess ||
        (t.zero != nullptr && (grp ? cudaMemset2DAsync(t.zero, BRL_PPO_SCRATCH_BYTES, 0, t.zero_bytes, (size_t)K, s)
                                   : cudaMemsetAsync(t.zero, 0, t.zero_bytes, s)) != cudaSuccess))
        return check_launch(t.what);
    // 1. minibatch gather of the observation (src/update.py:194-199, cast of src/update.py:95); a group's learner k reads
    //    row k of the trajectory table
    {
        const unsigned grid = (unsigned)(((int64_t)B * (kObsDimM / 8) + 255) / 256);
        uint16_t* o = reinterpret_cast<uint16_t*>(sc + S.obs);
        auto gather = [&](auto type) {
            using T = decltype(type);
            if (grp) launch_pdl(k_gather_obs_grouped<T>, dim3(grid, (unsigned)K), dim3(256), 0, s, grp->traj, (int64_t)B, o, (long long)S.total);
            else launch_pdl(k_gather_obs<T>, dim3(grid), dim3(256), 0, s, static_cast<const T*>(t.obs), t.index, (int64_t)B, o);
        };
        if (t.obs_flags & BRL_PPO_OBS_BF16) gather(__nv_bfloat16{});
        else if (t.obs_flags & BRL_PPO_OBS_U8) gather(uint8_t{});
        else gather(float{});
    }
    // 2. forward GEMMs; a group's as one launch over all learners' tiles, described by learner 0's ops
    OpSpec fwd[5], bwd[kMaxOps];
    const int nb = train_ops(fwd, bwd, sc, t.blob, grads, t.grad_sumsq, B);
    const GroupSpec gs{K, (long long)S.total, (long long)train_blob().total, (long long)param_stride(), BRL_PPO_SCRATCH_BYTES / (long long)sizeof(double)};
    const GroupSpec* g = grp ? &gs : nullptr;
    unsigned long long* trace = (t.tune & 8) ? reinterpret_cast<unsigned long long*>(sc + S.trace) : nullptr;  // tune bit 3
    // Tile widths, measured on B200 at B = 1024 (scripts/exp_train_trace.py): the forward is a chain of layers with one tile
    // per SM per layer, where 128 x 64 tiles win; the backward has two independent GEMMs per layer (dgrad, wgrad) to fill the
    // SMs, where 128 x 128 tiles move a third fewer operand bytes.  Tune bit 2 / bit 4 flip them.
    const bool wide_fwd = (t.tune & 4) != 0, wide_bwd = (t.tune & 16) == 0;
    if ((rc = launch_gemms(wide_fwd, s, fwd, 5, nmb, ready, trace, t.what, g)) != BRL_OK) return rc;
    if ((rc = check_launch(t.what)) != BRL_OK) return rc;
    // 3. the caller's loss head (and its backward into d loss / d (logits, value)), given learner 0's buffers
    TrainHeadIO io{};
    io.logits = reinterpret_cast<const float*>(sc + S.logits);
    io.value = reinterpret_cast<const float*>(sc + S.value);
    io.dlogits = reinterpret_cast<float*>(sc + S.dlogits);
    io.dvalue = reinterpret_cast<float*>(sc + S.dvalue);
    io.dz_hi = sc + S.dz5_hi;
    io.dz_lo = sc + S.dz5_lo;
    if ((rc = t.loss_head(s, io, t.ctx)) != BRL_OK) return rc;
    if (grads == nullptr) return BRL_OK;
    // 4. backward GEMMs
    rc = launch_gemms(wide_bwd, s, bwd, nb, nmb, ready + (size_t)kMaxOps * K * (nmb + 1), trace ? trace + (size_t)kTraceTiles * 8 : nullptr,
                      t.what, g);
    if (rc != BRL_OK) return rc;
    // 5. bias gradients (and the deferred illegal-action statistic)
    BiasArgs a{};
    for (int l = 0; l < 4; ++l) { a.hi[l] = bf(S.dz_hi[l]); a.lo[l] = bf(S.dz_lo[l]); }
    a.dlogits = io.dlogits;
    a.dvalue = io.dvalue;
    a.grads = grads; a.B = B; a.F = F;
    if (grp) {
        GroupedBiasArgs ga{};
        ga.a = a;
        ga.traj = grp->traj;
        ga.coefs = grp->coefs;
        ga.logits = io.logits;
        ga.stats = grp->stats;
        ga.acc = static_cast<unsigned char*>(t.zero);
        ga.sc_stride = (long long)S.total;
        ga.illegal_stat = grp->illegal_stat;
        ga.n_gram = gram_blocks(B, 1024);
        launch_pdl(k_bias_grad_grouped, dim3(4 * (kHidden / 64) + 1 + (grp->illegal_stat ? 1 : 0), (unsigned)K), dim3(1024), 0, s, ga);
    } else {
        a.sumsq = t.grad_sumsq;
        a.n_gram = t.gram ? t.n_gram : 0;
        if (a.n_gram) a.gram = *t.gram;
        launch_pdl(k_bias_grad, dim3(4 * (kHidden / 64) + 1 + (a.n_gram ? 1 : 0)), dim3(1024), 0, s, a);
    }
    return check_launch(t.what);
}

int32_t brl::sl_params_minibatch(const char* what, bool backward, cudaStream_t s, void** b, const void* opaque, size_t len,
                                 const SlParamsHead& head) {
    if (opaque == nullptr || len != sizeof(BrlSlParams))
        return fail(BRL_E_OPAQUE, "%s: opaque must be one BrlSlParams (%zu bytes), got %zu", what, sizeof(BrlSlParams), len);
    const BrlSlParams* p = static_cast<const BrlSlParams*>(opaque);
    if (p->batch < 0 || p->batch > (1 << 24)) return fail(BRL_E_OPAQUE, "%s: batch must be in [0, 2^24]", what);
    if (p->batch == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL
    const int grads = 3 + head.n_in, stats = grads + (backward ? 1 : 0), acc = stats + 1;  // buffer indices
    const char* names[16] = {"obs", "blob", "scratch"};
    for (int k = 0; k < head.n_in; ++k) names[3 + k] = head.in_names[k];
    if (backward) names[grads] = "grads";
    names[stats] = "stats";
    names[acc] = "acc";
    const int32_t rc = check_buffers(what, b, names, acc + 1, 0, 1u << 0 | 1u << 1 | 1u << 2 | (backward ? 1u << grads : 0u) | 1u << acc);
    if (rc != BRL_OK) return rc;
    for (int k = 0; k < head.n_in; ++k)
        if (((head.in_aligned4 >> k) & 1u) && (reinterpret_cast<uintptr_t>(b[3 + k]) & 3u) != 0)
            return fail(BRL_E_BUFFER, "%s: %s is not 4-byte aligned", what, head.in_names[k]);
    const SlHeadCtx ctx{b + 3, static_cast<float*>(b[stats]), static_cast<double*>(b[acc]), p->batch, p->ent_coef, backward};
    const int32_t tiles = p->flags & head.tile_flags;
    TrainMinibatch t{};
    t.obs = b[0];
    t.obs_flags = p->flags & (BRL_F_OBS_U8 | BRL_F_OBS_BF16);  // same bits as BRL_PPO_OBS_U8 / BRL_PPO_OBS_BF16
    t.tune = (tiles & BRL_CV_WIDE_FORWARD ? 4 : 0) | (tiles & BRL_CV_NARROW_BACKWARD ? 16 : 0);  // BrlPpoParams.reserved's bits
    t.batch = p->batch;
    t.blob = static_cast<const unsigned char*>(b[1]);
    t.scratch = static_cast<unsigned char*>(b[2]);
    t.grads = backward ? static_cast<float*>(b[grads]) : nullptr;
    t.grad_sumsq = backward ? ctx.acc + 14 : nullptr;
    t.zero = ctx.acc;
    t.zero_bytes = 16 * sizeof(double);
    t.what = what;
    t.loss_head = head.launch;
    t.ctx = &ctx;
    return launch_train_minibatch(s, t);
}
