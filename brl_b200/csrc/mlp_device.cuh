// mlp_device.cuh -- pieces shared by the tensor-core policy forward (brl_mlp.cu) and the PPO-update
// forward/backward GEMMs (brl_mlp_train.cu): tile constants, the packed-parameter layout, the TMA / tcgen05 /
// mbarrier PTX wrappers, the UMMA descriptors, the head-tile epilogue and the tensor-map encoder.  sm_100a only.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.h"

namespace brl {

constexpr int kObsDimM = 480, kHidden = 1024, kHeadValid = 39, kHeadPad = 64;
constexpr int kBM = 128, kBK = 64, kUmmaK = 16;
constexpr int kMlpThreads = 192;
constexpr uint32_t kSmemBudget = 200 * 1024;

// ---- packed parameter blob ---------------------------------------------------------------
struct MlpLayout {
    size_t w_hi[5], w_lo[5], bias[5], total;
    int n_out[5], k_in[5];
};

__host__ __device__ inline MlpLayout mlp_layout() {
    MlpLayout L{};
    size_t off = 0;
    for (int l = 0; l < 5; ++l) {
        L.k_in[l] = l == 0 ? kObsDimM : kHidden;
        L.n_out[l] = l == 4 ? kHeadPad : kHidden;
        size_t wbytes = (size_t)L.n_out[l] * L.k_in[l] * 2;
        L.w_hi[l] = off; off += wbytes;
        L.w_lo[l] = off; off += wbytes;
        L.bias[l] = off; off += (size_t)L.n_out[l] * 4;
        off = (off + 255) & ~(size_t)255;
    }
    L.total = off;
    return L;
}

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// bounded spin: a protocol bug becomes a trap (CUDA error), never a hung GPU
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    for (uint32_t it = 0; !done; ++it) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (it > (1u << 26)) __trap();
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
// shared -> global tile store through the TMA (bulk async-group completion)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }  // sources reusable
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }            // writes performed
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {  // implies tcgen05.fence::before_thread_sync
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major operand tile in shared memory, rows of 64 bf16 = 128 bytes, 128B swizzle, 8-row
// groups 1024 bytes apart (what the TMA box {64, rows} with CU_TENSOR_MAP_SWIZZLE_128B writes)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);      // start address, 16-byte units
    d |= (uint64_t)(1024u >> 4) << 32;                     // stride byte offset between 8-row groups
    d |= (uint64_t)1 << 46;                                // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                                // SWIZZLE_128B
    return d;
}
// kind::f16 instruction descriptor: bf16 x bf16 -> f32, both operands K-major, M x N tile
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// MN-major operand tile: the M (or N) index is the contiguous one, as when a [K, M] row-major matrix is staged by
// TMA boxes of {64 M-elements = 128 bytes, K rows} with 128B swizzle.  Canonical form (128-bit units):
// Swizzle<3,4,3> o ((8, m), (8, k)) : ((1, LBO), (8, SBO)): K rows 128 bytes apart, 8-row K groups SBO = 1024 bytes apart,
// 64-element M chunks LBO bytes apart (= the size of one staged box).  Advancing K by 16 = +2048 bytes on the start address.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t saddr, uint32_t lbo_bytes) {
    uint64_t d = (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;     // leading byte offset between 64-element MN chunks
    d |= (uint64_t)(1024u >> 4) << 32;                     // stride byte offset between 8-row K groups
    d |= (uint64_t)1 << 46;                                // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                                // SWIZZLE_128B
    return d;
}
// ... and the instruction descriptor with both operands MN-major (a_major, b_major = bits 15, 16)
__host__ __device__ constexpr uint32_t umma_idesc_bf16_mn(int m, int n) { return umma_idesc_bf16(m, n) | (1u << 15) | (1u << 16); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}

// head tile: columns 0..37 = policy logits, 38 = value (src/models.py:30-32)
__device__ __forceinline__ void epilogue_head_row(uint32_t t_row, const float* __restrict__ bias, bool row_ok,
                                                  float* __restrict__ logits_row, float* __restrict__ value_row) {
    uint32_t r0[32], r1[32];
    tmem_ld32(t_row, r0);
    tmem_ld32(t_row + 32u, r1);
    if (row_ok) {
        float2* pl = reinterpret_cast<float2*>(logits_row);
#pragma unroll
        for (int jj = 0; jj < 16; ++jj)
            pl[jj] = make_float2(__uint_as_float(r0[2 * jj]) + __ldg(bias + 2 * jj),
                                 __uint_as_float(r0[2 * jj + 1]) + __ldg(bias + 2 * jj + 1));
#pragma unroll
        for (int jj = 0; jj < 3; ++jj)
            pl[16 + jj] = make_float2(__uint_as_float(r1[2 * jj]) + __ldg(bias + 32 + 2 * jj),
                                      __uint_as_float(r1[2 * jj + 1]) + __ldg(bias + 32 + 2 * jj + 1));
        *value_row = __uint_as_float(r1[6]) + __ldg(bias + 38);
    }
}

// ---- host side --------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// bf16 matrix [rows, cols] row-major (row pitch `pitch` elements), box = 64 columns x box_rows, 128B swizzle;
// out-of-bounds elements read as zero (K tail of the 480-wide first layer, M / N tails)
static bool make_map(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t pitch, uint32_t box_rows) {
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {pitch * 2};
    cuuint32_t box[2] = {(cuuint32_t)kBK, box_rows};
    cuuint32_t estr[2] = {1, 1};
    return encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// bf16 matrix [rows, cols] row-major as the DESTINATION of epilogue stores: box = 32 columns (64 bytes) x 32 rows with the
// 64-byte swizzle, i.e. the 2 KB block one epilogue warp stages per 32-column chunk (lane = row).  Rows past `rows` are clipped.
static bool make_map_store(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint64_t pitch) {
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {pitch * 2};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t estr[2] = {1, 1};
    return encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// general bf16 tensor map (rank <= 5), 128B swizzle, zero fill: dims / box innermost first, strides in bytes for dims 1..
static inline bool make_map_nd(CUtensorMap* m, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box) {
    cuuint64_t d[5], s[4];
    cuuint32_t b[5], e[5] = {1, 1, 1, 1, 1};
    for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; }
    for (int i = 0; i + 1 < rank; ++i) s[i] = strides_bytes[i];
    return encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(ptr), d, s, b, e, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace brl
