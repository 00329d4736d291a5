// common.h -- error plumbing shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>

#include "../../include/brl_b200.h"

namespace brl {

char* last_error_buffer();  // thread-local, 512 bytes

inline int32_t fail(int32_t code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(last_error_buffer(), 512, fmt, ap);
    va_end(ap);
    return code;
}

inline int32_t check_launch(const char* what) {
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return fail(BRL_E_LAUNCH, "%s: %s", what, cudaGetErrorString(err));
    return BRL_OK;
}

inline const BrlParams* get_params(const void* opaque, size_t opaque_len, int32_t* rc) {
    if (opaque == nullptr || opaque_len != sizeof(BrlParams)) {
        *rc = fail(BRL_E_OPAQUE, "opaque must be one BrlParams (%zu bytes), got %zu", sizeof(BrlParams), opaque_len);
        return nullptr;
    }
    const BrlParams* p = static_cast<const BrlParams*>(opaque);
    if (p->n_envs < 0) {
        *rc = fail(BRL_E_OPAQUE, "n_envs < 0");
        return nullptr;
    }
    *rc = BRL_OK;
    return p;
}

// Per-device slot of a function-local cache (SM count, "kernel attribute already set", co-resident CTA count): these are
// per-device facts, and a process may drive several GPUs.  Races only repeat idempotent driver calls.
constexpr int kMaxDevices = 64;
inline int device_slot() {
    int dev = 0;
    cudaGetDevice(&dev);
    return dev >= 0 && dev < kMaxDevices ? dev : 0;
}

// SM count of the current device, which sizes the persistent grids (148 on a B200 if the query fails)
inline int sm_count() {
    static int n_sm_dev[kMaxDevices] = {};
    int& n_sm = n_sm_dev[device_slot()];
    if (n_sm == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n_sm <= 0) n_sm = 148;
    }
    return n_sm;
}

// Grouped forward over a pool of nets (brl_model_rows -> brl_policy_act_grouped): each net's rows are padded to this height,
// the row tile of the fused forward's CTA pairs, so that no tile mixes two nets.
constexpr int kGroupRows = 256;

// batches from this size on run the policy forward as one fused launch on CTA pairs (brl_mlp.cu fused_forward; also the rule
// brl_duplicate_match's device loop applies to its device-side row count)
constexpr int kPairMinM = 4096;

// masked categorical over f32 logits[n,38] (brl_algo.cu); shared by brl_categorical and the unfused brl_policy_act path
int32_t launch_categorical(cudaStream_t stream, const float* logits, const unsigned char* mask, int32_t* action, float* log_prob,
                           int64_t n, int sample, uint64_t seed, int64_t env_offset, uint32_t step, const int32_t* row_index = nullptr,
                           float* logits_by_env = nullptr);

// brl_ppo_loss's body (brl_ppo.cu), optionally also writing d loss / d (logits, value) as bf16 hi / lo rows [B, 64] for brl_ppo_grad
// acc_zeroed: the caller already cleared the f64[16] scratch on this stream (keeps a memset out of a PDL kernel chain)
// defer_illegal (honoured only when illegal_l2_coef == 0): only the partial Gram matrices are formed before the loss kernel;
// the caller runs gram_tail() itself later (brl_ppo_grad: a spare block of k_bias_grad) with gram_args(buffers, p, &stats[6])
// and gram_blocks(batch, 1024) partials
// anchor (brl_ppo_grad_anchored): also the KL term to a fixed reference policy (stats[7] = its mean over the minibatch)
struct PpoAnchor {
    const float* logits;     // f32 [total, 38]: the anchor's logits in the rows of the flat trajectory (solo)
    const long long* table;  // [K] device addresses of each learner's anchor logits (grouped; NULL = solo)
    const float* coef;       // f32 kl_coef: [1] solo, [K] grouped (device scalars)
};
int32_t launch_ppo_loss(cudaStream_t stream, void** buffers, const BrlPpoParams* p, void* dz_hi, void* dz_lo, bool acc_zeroed,
                        bool defer_illegal, const PpoAnchor* anchor = nullptr);
struct GramArgs;
GramArgs gram_args(void** loss_buffers, const BrlPpoParams* p, float* stat);
int gram_blocks(int64_t batch, int threads);

// One minibatch through the DeepMind MLP on tcgen05 (brl_mlp_train.cu), shared by brl_ppo_grad, brl_sl_grad /
// brl_sl_eval and brl_cv_grad / brl_cv_eval: gather of the observation, fused forward with the activations kept, the caller's loss head, then (when
// `grads` is set) the fused backward and the bias sums.  The ops differ only in the loss head.
struct TrainHeadIO {  // what the forward leaves for the loss head, and where the backward reads d loss / d (logits, value)
    const float* logits;  // f32 [B, 38]
    const float* value;   // f32 [B]
    float* dlogits;       // f32 [B, 38] (the head's bias sums read it)
    float* dvalue;        // f32 [B]
    void* dz_hi;          // bf16 hi / lo [B, 64]: 38 logits, value, zeros (the head's dgrad / wgrad operand)
    void* dz_lo;
};
// K learners in the launches of one minibatch (brl_ppo_grad_grouped), learner 0's buffers in TrainMinibatch: learner k's
// scratch lies k * train_scratch(batch).total bytes further, its blob k * brl_mlp_train_blob_bytes(), its grads
// k * brl_mlp_param_stride() floats, its accumulators (`zero`, `grad_sumsq`) k * BRL_PPO_SCRATCH_BYTES bytes; the grouped
// tile counters follow the K scratches.  `obs` and `index` are unused: they come from the trajectory table.
struct TrainGroup {
    int K;
    const long long* traj;  // [K][8] (ops.ppo_trajectory_row): the gather reads obs and index, the Gram tail index and mask
    const float* coefs;     // [K][4]: the Gram tail runs for a learner whose illegal_l2_coef (column 3) is 0
    float* stats;           // [K][8]
    bool illegal_stat;      // BRL_PPO_ILLEGAL_STAT
};
struct TrainMinibatch {
    const void* obs;             // [total, 480] f32, or u8 / bf16 with obs_flags BRL_PPO_OBS_U8 / BRL_PPO_OBS_BF16
    int32_t obs_flags;
    const int32_t* index;        // [B] rows of obs, NULL = identity
    int64_t batch;
    const unsigned char* blob;   // brl_mlp_pack_train
    unsigned char* scratch;      // brl_mlp_train_scratch_bytes(batch)
    float* grads;                // flat fp32 gradient, NULL = forward and loss head only
    double* grad_sumsq;          // += |grads|^2, or NULL
    void* zero;                  // caller's accumulators, cleared together with the tile counters (NULL = none)
    size_t zero_bytes;
    int32_t tune;                // BrlPpoParams.reserved bits
    const GramArgs* gram;        // deferred illegal-probability statistic, tail run in a spare block of the bias sums
    int n_gram;                  // (0 = none)
    const char* what;            // op name for error messages
    int32_t (*loss_head)(cudaStream_t, const TrainHeadIO&, const void* ctx);
    const void* ctx;
    const TrainGroup* group;     // NULL = one learner
};
int32_t launch_train_minibatch(cudaStream_t stream, const TrainMinibatch& t);

// Grid of a warp-per-sample loss head (128 threads, 4 samples a block): one sample per warp, at most 8 blocks per SM of a B200
inline unsigned head_grid(int64_t batch) {
    const unsigned grid = (unsigned)((batch + 3) / 4);
    return grid > 148u * 8u ? 148u * 8u : grid;
}

// The ops whose opaque is a BrlSlParams (brl_sl_grad / brl_sl_eval, brl_cv_grad / brl_cv_eval): one minibatch through
// launch_train_minibatch with the head's kernel.  Buffers: [0] obs [1] blob [2] scratch, the head's n_in inputs, then
// grads (backward only), stats, acc.  obs, blob, scratch, grads and acc are 16-byte aligned.
struct SlParamsHead {
    int n_in;              // at most 10
    const char* const* in_names;
    unsigned in_aligned4;  // bit k: input k must be 4-byte aligned
    int32_t tile_flags;    // BrlSlParams.flags bits the op honours: BRL_CV_WIDE_FORWARD / BRL_CV_NARROW_BACKWARD
    int32_t (*launch)(cudaStream_t, const TrainHeadIO&, const void* ctx);  // ctx: the SlHeadCtx below
};
struct SlHeadCtx {
    void* const* in;  // the head's input buffers
    float* stats;     // [8]
    double* acc;      // f64[16], cleared before the forward: the head's sums from 0, |grads|^2 at 14, its ticket at 15
    int64_t B;
    float ent_coef;
    bool backward;    // d loss / d (logits, value) wanted (brl_*_grad)
};
int32_t sl_params_minibatch(const char* what, bool backward, cudaStream_t stream, void** buffers, const void* opaque, size_t len,
                            const SlParamsHead& head);

// brl_ppo_grad_grouped's loss head (brl_ppo.cu): launch_ppo_loss for K learners, one grid row per learner.  Learner k's
// trajectory buffers are row k of the device table `traj`, its coefficients row k of `coefs`; its forward outputs and
// d loss buffers lie k * sc_stride bytes after learner 0's `head`, its stats at stats + 8k, its f64 accumulators (cleared
// by the caller) at acc + k * BRL_PPO_SCRATCH_BYTES.  A zero illegal_l2_coef defers the logged statistic to the bias sums.
struct PpoGroupIO {
    const long long* traj;  // [K][8]: obs, index, mask, action, old_log_prob, old_value, advantages, targets
    const float* coefs;     // [K][4]: clip_eps, ent_coef, vf_coef, illegal_l2_coef
    TrainHeadIO head;
    long long sc_stride;
    float* stats;
    unsigned char* acc;
    int64_t batch;
    int K;
    int32_t flags;
    const PpoAnchor* anchor;  // brl_ppo_grad_grouped_anchored (NULL: no KL term)
};
int32_t launch_ppo_loss_grouped(cudaStream_t stream, const PpoGroupIO& io);

// Programmatic dependent launch for the short kernels of a dependent chain (the PPO optimizer step): the kernel may be
// scheduled while its predecessor in the stream drains; it must execute pdl_wait() before touching global memory and
// should call pdl_trigger() first so that ITS successor can be scheduled early too.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute at{};
    at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

#define BRL_REQUIRE(ptr, name)                                                            \
    do {                                                                                  \
        if ((ptr) == nullptr) return brl::fail(BRL_E_BUFFER, "%s: buffer '%s' is NULL", __func__, name); \
        if ((reinterpret_cast<uintptr_t>(ptr) & 15u) != 0)                                \
            return brl::fail(BRL_E_BUFFER, "%s: buffer '%s' is not 16-byte aligned", __func__, name);    \
    } while (0)

// An op's buffer checks, in buffer order: b[k] must not be NULL unless bit k of `nullable` is set, and must be 16-byte
// aligned when bit k of `aligned16` is set, else align[k]-byte aligned when `align` is given (0 or 1: any address).  `what`
// names the op in the message.
inline int32_t check_buffers(const char* what, void* const* b, const char* const* names, int n, unsigned nullable, unsigned aligned16,
                             const uint8_t* align = nullptr) {
    for (int k = 0; k < n; ++k) {
        if (b[k] == nullptr && !((nullable >> k) & 1u)) return fail(BRL_E_BUFFER, "%s: buffer '%s' is NULL", what, names[k]);
        const unsigned a = (aligned16 >> k) & 1u ? 16u : align != nullptr && align[k] > 1 ? align[k] : 1u;
        if ((reinterpret_cast<uintptr_t>(b[k]) & (a - 1)) != 0)
            return fail(BRL_E_BUFFER, "%s: buffer '%s' is not %u-byte aligned", what, names[k], a);
    }
    return BRL_OK;
}

}  // namespace brl
