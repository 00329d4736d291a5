// ppo_gram.cuh -- illegal_action_loss = ||P * ~mask||_2 / 2 with P = softmax(logits) [B, 38] (src/update.py:138-142).
// jnp.linalg.norm(.., ord=2) of a 2-D array is the SPECTRAL norm: the largest singular value sigma_1 of X = P * ~mask.
// sigma_1^2 is the top eigenvalue of the 38 x 38 Gram matrix G = X^T X, and d sigma_1 / d X = u_1 v_1^T with v_1 its
// eigenvector and u_1 = X v_1 / sigma_1, so the loss kernel needs only (sigma_1, v_1).
//
// gram_partial<T>(): ONE block (T threads) of n_blocks (<= kGramBlocks) forms the partial Gram matrix of its samples (x rows
// staged in shared memory, every thread owns entries of X^T X) and stores it.  gram_tail(): one block sums the partials
// and one warp runs power iteration on the fp32 G from the start G.1 (X >= 0, so v_1 >= 0 and the start has a large
// component along it), 8 steps between convergence checks, until v stops moving (<= tol: 1e-6 when v_1 feeds the gradient,
// 3e-4 when only sigma_1 is wanted) or 160 steps; sigma_1 = sqrt of the double Rayleigh quotient (second order in the
// remaining direction error, so 3e-4 in v leaves ~1e-7 in sigma_1).  (Six normalised squarings of G, tried
// first -- fp32 SIMT tiles, then 3xTF32 mma.sync -- cost ~3,500 SM clocks EACH on B200 against ~200 for a matvec step:
// scripts/exp_gram_phases.py.)
// k_ppo_illegal_gram (brl_ppo.cu) runs both before the loss kernel, which then has sigma_1 / v_1 for the gradient.  When the
// coefficient is 0 only the logged statistic needs the norm: brl_ppo_grad then runs only the partials before the loss
// kernel (k_ppo_gram_partial) and the serial tail as one spare block of k_bias_grad (brl_mlp_train.cu), beside the bias
// sums.  (Also tried, scripts/exp_gram_cost.py: the partials as extra blocks of the loss launch -- they outlast the loss
// blocks; the whole computation as a side kernel the backward launch does not wait for -- no overlap was observed.)
#pragma once
#include <math.h>
#include <stdint.h>

namespace brl {

constexpr int kGramA = 38, kGramPad = 40, kGramBlocks = 16, kGramN = kGramA * kGramA;
constexpr int kGramLd = 39;  // row stride of the fp32 G in shared memory: odd, so lane = row reads are conflict-free

struct GramArgs {
    const float* logits;    // [B, 38]
    const int32_t* index;   // [B] rows of the flat trajectory (NULL = identity)
    const uint8_t* mask;    // [total, 38]
    int64_t B;
    unsigned long long* ticket;  // zeroed before the launch
    double* spec;           // out [40]: sigma_1, v_1[38], 0
    float* part;            // scratch [kGramBlocks][38 * 38]
    float* stat;            // out: illegal_action_loss = sigma_1 / 2 (NULL: the caller forms it from spec)
    float tol;              // power iteration stops when no component of v moved by more than this over 8 steps
};

// GramArgs of one minibatch whose f64 accumulators are `acc` (BRL_PPO_SCRATCH_BYTES: the ticket is f64 13, the spectrum
// starts at byte 128, the partials at byte 512); stat != NULL: the statistic alone is wanted
__host__ __device__ inline GramArgs gram_args_at(const float* logits, const int32_t* index, const uint8_t* mask, int64_t B,
                                                 unsigned char* acc, float* stat) {
    GramArgs g{};
    g.logits = logits;
    g.index = index;
    g.mask = mask;
    g.B = B;
    g.ticket = reinterpret_cast<unsigned long long*>(acc + 13 * sizeof(double));
    g.spec = reinterpret_cast<double*>(acc + 128);
    g.part = reinterpret_cast<float*>(acc + 512);
    g.stat = stat;
    g.tol = stat ? 3e-4f : 1e-6f;  // statistic only (deferred) vs v_1 feeding the loss gradient
    return g;
}

struct GramSmem {
    float X[64 * kGramPad];        // staging of 64 sample rows (gram_partial<1024>)
    double Gd[kGramN];             // G in double (final Rayleigh quotient)
    float Gf[kGramA * kGramLd];    // G in float (power iteration)
    float vec[kGramPad];
    float red[32];
    int last;
};

__device__ __forceinline__ float gram_block_sum(GramSmem& sm, float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sm.red[threadIdx.x >> 5] = v;
    __syncthreads();
    float t = 0.0f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sm.red[w];
    return t;
}

// Partial Gram matrix of the samples of block `block` out of `n_blocks`, no atomics: chunks of 2 samples per warp leave
// their illegal-probability rows x in shared memory (Xs: [2 * kThreads / 32][kGramPad] floats), then every thread
// accumulates its entries (tid, tid + kThreads, ...) of X^T X in registers and stores them to a.part[block].
template <int kThreads>
__device__ __forceinline__ void gram_partial(const GramArgs& a, int block, int n_blocks, float* Xs) {
    constexpr int kWarps = kThreads / 32, kChunk = 2 * kWarps, kPer = (kGramN + kThreads - 1) / kThreads;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float (*X)[kGramPad] = reinterpret_cast<float (*)[kGramPad]>(Xs);
    float acc[kPer];
    int ei[kPer], ej[kPer];
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
        const int e = tid + k * kThreads < kGramN ? tid + k * kThreads : 0;
        acc[k] = 0.0f; ei[k] = e / kGramA; ej[k] = e % kGramA;
    }
    const bool in1 = lane < kGramA - 32;
    for (int64_t base = (int64_t)block * kChunk; base < a.B; base += (int64_t)n_blocks * kChunk) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int s = warp * 2 + k;
            const int64_t b = base + s;
            float x0 = 0.0f, x1 = 0.0f;
            if (b < a.B) {
                const int64_t src = a.index ? a.index[b] : b;
                const float l0 = a.logits[b * kGramA + lane], l1 = in1 ? a.logits[b * kGramA + 32 + lane] : -INFINITY;
                const bool ill0 = a.mask[src * kGramA + lane] == 0, ill1 = in1 && a.mask[src * kGramA + 32 + lane] == 0;
                float mx = fmaxf(l0, l1);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                const float ex0 = expf(l0 - mx), ex1 = in1 ? expf(l1 - mx) : 0.0f;
                float se = ex0 + ex1;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
                const float lse = mx + logf(se);
                x0 = ill0 ? expf(l0 - lse) : 0.0f;  // as Row::softmax (brl_ppo.cu)
                x1 = ill1 ? expf(l1 - lse) : 0.0f;
            }
            X[s][lane] = x0;
            if (in1) X[s][32 + lane] = x1;
        }
        __syncthreads();
#pragma unroll 4
        for (int s = 0; s < kChunk; ++s)
#pragma unroll
            for (int k = 0; k < kPer; ++k) acc[k] = fmaf(X[s][ei[k]], X[s][ej[k]], acc[k]);
        __syncthreads();
    }
    float* part = a.part + (size_t)block * kGramN;
#pragma unroll
    for (int k = 0; k < kPer; ++k)
        if (tid + k * kThreads < kGramN) part[tid + k * kThreads] = acc[k];
}

#ifdef BRL_GRAM_TIMING
#define BRL_GRAM_STAMP(i) do { if (threadIdx.x == 0) reinterpret_cast<long long*>(a.spec + 40)[i] = clock64(); } while (0)
#else
#define BRL_GRAM_STAMP(i)
#endif

// The serial part, one block (any multiple of 32 threads), after all n_blocks partials are visible.
__device__ __forceinline__ void gram_tail(const GramArgs& a, int n_blocks, GramSmem& sm) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    BRL_GRAM_STAMP(0);
    // G = sum of the partials (fp32 adds of <= 32 non-negative terms; kept in double for the final Rayleigh quotient)
    float tr_local = 0.0f;
    for (int k = tid; k < kGramN; k += blockDim.x) {
        float sum = 0.0f;
#pragma unroll
        for (int half = 0; half < kGramBlocks / 16; ++half) {
            float v[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int blk = 16 * half + q;
                v[q] = blk < n_blocks ? __ldcg(a.part + (size_t)blk * kGramN + k) : 0.0f;
            }
#pragma unroll
            for (int q = 0; q < 16; ++q) sum += v[q];
        }
        sm.Gd[k] = (double)sum;
        sm.Gf[(k / kGramA) * kGramLd + k % kGramA] = sum;
        if (k / kGramA == k % kGramA) tr_local += sum;
    }
    BRL_GRAM_STAMP(1);
    const float tr = gram_block_sum(sm, tr_local);
    if (!(tr > 0.0f)) {  // no probability mass on illegal actions in this minibatch
        if (tid < 40) a.spec[tid] = 0.0;
        if (tid == 0 && a.stat) *a.stat = 0.0f;
        return;
    }
    BRL_GRAM_STAMP(2);
    if (warp != 0) return;
    // one warp: lane l owns rows l and (l < 6) 32 + l
    const bool in1 = lane < kGramA - 32;
    const float* g0 = &sm.Gf[lane * kGramLd];
    const float* g1 = &sm.Gf[(in1 ? 32 + lane : 0) * kGramLd];
    auto matvec = [&](float& v0, float& v1) {  // (v0, v1) <- G (v0, v1); the vector is exchanged through sm.vec
        __syncwarp();
        sm.vec[lane] = v0;
        if (in1) sm.vec[32 + lane] = v1;
        __syncwarp();
        float a0 = 0.0f, b0 = 0.0f, a1 = 0.0f, b1 = 0.0f;
#pragma unroll
        for (int m = 0; m < kGramA; m += 2) {
            const float va = sm.vec[m], vb = sm.vec[m + 1];
            a0 = fmaf(g0[m], va, a0);
            b0 = fmaf(g0[m + 1], vb, b0);
            a1 = fmaf(g1[m], va, a1);
            b1 = fmaf(g1[m + 1], vb, b1);
        }
        v0 = a0 + b0;
        v1 = in1 ? a1 + b1 : 0.0f;
    };
    auto normalise = [&](float& v0, float& v1) {
        float nn = v0 * v0 + v1 * v1;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) nn += __shfl_xor_sync(0xffffffffu, nn, o);
        const float rn = rsqrtf(nn);
        v0 *= rn; v1 *= rn;
    };
    float v0 = 1.0f, v1 = in1 ? 1.0f : 0.0f;
    matvec(v0, v1);  // start: G . 1
    normalise(v0, v1);
    for (int round = 0; round < 20; ++round) {
        const float p0 = v0, p1 = v1;
#pragma unroll 1
        for (int it = 0; it < 8; ++it) {
            matvec(v0, v1);
            if (it == 3) normalise(v0, v1);  // lambda_1 <= B: four unnormalised steps stay far inside the fp32 range
        }
        normalise(v0, v1);
        float d = fmaxf(fabsf(v0 - p0), fabsf(v1 - p1));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d = fmaxf(d, __shfl_xor_sync(0xffffffffu, d, o));
        if (d <= a.tol) break;
    }
    BRL_GRAM_STAMP(3);
    __syncwarp();
    sm.vec[lane] = v0;
    if (in1) sm.vec[32 + lane] = v1;
    __syncwarp();
    BRL_GRAM_STAMP(4);
    // (v0, v1) = unit v_1 (fp32); sigma_1^2 = v^T G v / v^T v in double
    double w0 = 0.0, w0b = 0.0, w1 = 0.0, w1b = 0.0;
#pragma unroll 2
    for (int m = 0; m < kGramA; m += 2) {
        const double va = (double)sm.vec[m], vb = (double)sm.vec[m + 1];
        w0 += sm.Gd[lane * kGramA + m] * va;
        w0b += sm.Gd[lane * kGramA + m + 1] * vb;
        if (in1) {
            w1 += sm.Gd[(32 + lane) * kGramA + m] * va;
            w1b += sm.Gd[(32 + lane) * kGramA + m + 1] * vb;
        }
    }
    double ray = (w0 + w0b) * (double)v0 + (w1 + w1b) * (double)v1, vv = (double)v0 * v0 + (double)v1 * v1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ray += __shfl_xor_sync(0xffffffffu, ray, o);
        vv += __shfl_xor_sync(0xffffffffu, vv, o);
    }
    BRL_GRAM_STAMP(5);
    const double sigma = sqrt(fmax(ray / vv, 0.0));
    a.spec[1 + lane] = (double)v0;
    if (in1) a.spec[33 + lane] = (double)v1;
    if (lane == 0) {
        a.spec[0] = sigma;
        a.spec[39] = 0.0;
        if (a.stat) *a.stat = 0.5f * (float)sigma;
    }
}

// partial + tail in one launch of n_blocks x kThreads threads: the last block to finish (ticket) runs the tail
template <int kThreads>
__device__ __forceinline__ void gram_block(const GramArgs& a, int block, int n_blocks, GramSmem& sm) {
    gram_partial<kThreads>(a, block, n_blocks, sm.X);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) sm.last = atomicAdd(a.ticket, 1ull) == (unsigned long long)n_blocks - 1ull;
    __syncthreads();
    if (!sm.last) return;
    __threadfence();
    gram_tail(a, n_blocks, sm);
}

}  // namespace brl
