// obs_row.cuh -- expansion of a 15-word observation bit row into one f32 / u8 / bf16 observation row, one warp per row.
// Shared by the env kernels (brl_env.cu) and the hand-reading expansion (brl_posterior.cu).
#pragma once
#include <stdint.h>

#include "env_device.cuh"

namespace brl {

enum ObsKind { kObsF32 = 0, kObsU8 = 1, kObsBF16 = 2 };

// 4 bits -> 4 bytes of 0/1
__device__ __forceinline__ uint32_t spread4(uint32_t nib) { return (nib * 0x00204081u) & 0x01010101u; }

__device__ __forceinline__ float4 nibble_to_float4(uint32_t nib) {
    return make_float4((nib & 1u) ? 1.0f : 0.0f, (nib & 2u) ? 1.0f : 0.0f, (nib & 4u) ? 1.0f : 0.0f,
                       (nib & 8u) ? 1.0f : 0.0f);
}

// 2 bits -> two bf16 (0x3F80 = 1.0) packed in one word
__device__ __forceinline__ uint32_t pair_to_bf16x2(uint32_t two) {
    return ((two & 1u) ? 0x00003F80u : 0u) | ((two & 2u) ? 0x3F800000u : 0u);
}

// phase 2 building blocks: cooperative, fully coalesced expansion.
// One warp writes one observation row (480 values) from its 15 words of bits.
template <int OBS>
__device__ __forceinline__ void emit_obs_row(const uint32_t* R, int lane, void* obs, int64_t env) {
    if (OBS == kObsF32) {
        float4* row = reinterpret_cast<float4*>(obs) + env * (kObsDim / 4);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int j = lane + 32 * k;
            if (j < kObsDim / 4) row[j] = nibble_to_float4((R[j >> 3] >> ((j & 7) * 4)) & 15u);
        }
    } else if (OBS == kObsU8) {
        uint4* row = reinterpret_cast<uint4*>(obs) + env * (kObsDim / 16);
        if (lane < kObsDim / 16) {
            uint32_t h = (R[lane >> 1] >> ((lane & 1) * 16)) & 0xFFFFu;
            row[lane] = make_uint4(spread4(h & 15u), spread4((h >> 4) & 15u), spread4((h >> 8) & 15u), spread4(h >> 12));
        }
    } else {
        uint4* row = reinterpret_cast<uint4*>(obs) + env * (kObsDim / 8);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            int j = lane + 32 * k;
            if (j < kObsDim / 8) {
                uint32_t b = (R[j >> 2] >> ((j & 3) * 8)) & 0xFFu;
                row[j] = make_uint4(pair_to_bf16x2(b), pair_to_bf16x2(b >> 2), pair_to_bf16x2(b >> 4), pair_to_bf16x2(b >> 6));
            }
        }
    }
}

}  // namespace brl
