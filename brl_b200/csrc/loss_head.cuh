// loss_head.cuh -- the device pieces of the warp-per-sample loss heads on the tensor-core training path (k_ppo_loss,
// k_sl_loss, k_cv_loss): one warp per sample, lane owning actions lane and lane + 32.
#pragma once
#include <cuda_bf16.h>
#include <math.h>

#include "common.h"

namespace brl {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// element idx of d loss / d (logits, value) as bf16 hi / lo (hi + lo = v to bf16 x bf16 precision): the operand of the
// head's input-gradient and weight-gradient GEMMs
__device__ __forceinline__ void store_dz(unsigned short* hi, unsigned short* lo, int64_t idx, float v) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v), l = __float2bfloat16_rn(v - __bfloat162float(h));
    hi[idx] = *reinterpret_cast<const unsigned short*>(&h);
    lo[idx] = *reinterpret_cast<const unsigned short*>(&l);
}

// softmax of the lane's logits l over the `sel` entries: returns the log-partition; p / logp = probabilities and their
// logs (0 / -inf outside sel)
__device__ __forceinline__ float softmax_sel(const float l[2], const bool sel[2], float p[2], float logp[2]) {
    const float mx = warp_max(fmaxf(sel[0] ? l[0] : -INFINITY, sel[1] ? l[1] : -INFINITY));
    const float lse = mx + logf(warp_sum((sel[0] ? expf(l[0] - mx) : 0.0f) + (sel[1] ? expf(l[1] - mx) : 0.0f)));
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        logp[k] = sel[k] ? l[k] - lse : -INFINITY;
        p[k] = sel[k] ? expf(logp[k]) : 0.0f;
    }
    return lse;
}

// One accumulator add: f64 sums, or int64 fixed-point sums kept in the f64 slots (exact, so independent of block order).
// Two overloads rather than a callable: passing the add as a lambda changes the heads' code.
__device__ __forceinline__ void acc_add(double* acc, double v) { atomicAdd(acc, v); }
__device__ __forceinline__ void acc_add(double* acc, long long v) {
    atomicAdd(reinterpret_cast<unsigned long long*>(acc), (unsigned long long)v);
}

// The tail of a 128-thread head: the four warps' lane-0 sums s[0..N) are added per block into acc[0..N) (one set of
// same-address atomics per block, not per warp), then each block takes a ticket in acc[ticket_slot].  Returns true in
// thread 0 of the last block to arrive, which then sees every block's sums and forms the statistics: no finalize launch.
template <int N, class T>
__device__ __forceinline__ bool head_block_sums(const T (&s)[N], double* acc, int ticket_slot) {
    __shared__ T part[4][N];
    __shared__ bool last_block;
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0)
        for (int k = 0; k < N; ++k) part[w][k] = s[k];
    __syncthreads();
    if (threadIdx.x < N) {
        const int k = threadIdx.x;
        acc_add(&acc[k], part[0][k] + part[1][k] + part[2][k] + part[3][k]);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long t = atomicAdd(reinterpret_cast<unsigned long long*>(&acc[ticket_slot]), 1ull);
        last_block = t == (unsigned long long)gridDim.x - 1ull;
    }
    __syncthreads();
    const bool last = last_block && threadIdx.x == 0;
    if (last) __threadfence();
    return last;
}

}  // namespace brl
