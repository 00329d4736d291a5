// brl_sl.cu -- supervised bidding pre-training (sl.py of the reference): the cross-entropy + masked-entropy loss head
// that rides on the tensor-core forward / backward of brl_mlp_train.cu.  (The examples, brl_sl_examples, are a tile kernel
// of brl_env.cu, next to the env kernels whose phase 2 they share.)
//
//   brl_sl_grad      value_and_grad(loss) (sl.py:169-184, 205-206) for one minibatch: launch_train_minibatch with k_sl_loss
//                    as the loss head.
//   brl_sl_eval      loss / accuracy / illegal-action probability (sl.py:169-194, 288-301) without the backward.
// The optimizer step is brl_mlp_adam_step with eps = 1e-8 and no clipping (optax.adam(learning_rate), sl.py:166).
#include <cuda_bf16.h>
#include <math.h>

#include "common.h"

namespace brl {

// ---- loss head -----------------------------------------------------------------------------------------------------
enum { kSlAccTarget = 0, kSlAccEnt, kSlAccCorrect, kSlAccIllegal, kSlAccSumsq = 14, kSlAccTicket = 15 };

struct SlLossArgs {
    const float* logits;  // [B, 38]
    const uint8_t* mask;  // [B, 38]
    const int32_t* label; // [B]
    float* dlogits;       // [B, 38] or NULL (brl_sl_eval)
    float* dvalue;        // [B]
    unsigned short* dz_hi;
    unsigned short* dz_lo;
    float* stats;         // [8]
    double* acc;          // [16], zeroed by the caller
    int64_t B;
    float ent_coef;
};

__device__ __forceinline__ float sl_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float sl_warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ void sl_split_store(const SlLossArgs& a, int64_t idx, float v) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v), l = __float2bfloat16_rn(v - __bfloat162float(h));
    a.dz_hi[idx] = *reinterpret_cast<const unsigned short*>(&h);
    a.dz_lo[idx] = *reinterpret_cast<const unsigned short*>(&l);
}

// stats = {total_loss, target_loss, entropy, accuracy, illegal_actions_prob, 0, 0, 0}; run by the last block
__device__ __forceinline__ void sl_finalize(const SlLossArgs& a) {
    const volatile double* acc = a.acc;
    const double B = (double)a.B;
    const float target = (float)(acc[kSlAccTarget] / (38.0 * B)), entropy = (float)(acc[kSlAccEnt] / B);
    a.stats[0] = target - a.ent_coef * entropy;
    a.stats[1] = target;
    a.stats[2] = entropy;
    a.stats[3] = (float)(acc[kSlAccCorrect] / B);
    a.stats[4] = (float)(acc[kSlAccIllegal] / B);
    a.stats[5] = a.stats[6] = a.stats[7] = 0.0f;
}

// One warp per sample, lane owns actions lane and lane + 32 (k_ppo_loss's layout).
//   target_loss = -mean(one_hot(label, 38) * log_softmax(logits))      over B * 38 entries, UNMASKED softmax (sl.py:178-179)
//   entropy     = mean of the entropy of softmax over the legal calls   (sl.py:180-182; select semantics, SURVEY 7)
//   total       = target_loss - ent_coef * entropy                      (sl.py:183)
//   d total / d logit_j = (q_j - [j == label]) / (38 B) + ent_coef * [legal j] p_j (log p_j + H) / B,  d total / d value = 0
//   accuracy    = mean(argmax softmax(logits) == label)                 (sl.py:186-194; first index on ties, as jnp.argmax)
//   illegal     = mean(softmax(logits) . ~legal)                        (sl.py:293-294)
__global__ void __launch_bounds__(128) k_sl_loss(const SlLossArgs a) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float inv38B = 1.0f / (38.0f * (float)a.B), invB = 1.0f / (float)a.B;
    double s_target = 0.0, s_ent = 0.0, s_correct = 0.0, s_ill = 0.0;
    for (int64_t b = warp; b < a.B; b += nw) {
        float l[2], q[2], p[2], logp[2];
        bool in[2], legal[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int j = lane + 32 * k;
            in[k] = j < BRL_NUM_ACTIONS;
            l[k] = in[k] ? a.logits[b * BRL_NUM_ACTIONS + j] : -INFINITY;
            legal[k] = in[k] && a.mask[b * BRL_NUM_ACTIONS + j] != 0;
        }
        const int label = a.label[b];
        // unmasked softmax
        const float mx = sl_warp_max(fmaxf(l[0], l[1]));
        const float lse = mx + logf(sl_warp_sum((in[0] ? expf(l[0] - mx) : 0.0f) + (in[1] ? expf(l[1] - mx) : 0.0f)));
#pragma unroll
        for (int k = 0; k < 2; ++k) q[k] = in[k] ? expf(l[k] - lse) : 0.0f;
        // softmax over the legal calls
        const float mxl = sl_warp_max(fmaxf(legal[0] ? l[0] : -INFINITY, legal[1] ? l[1] : -INFINITY));
        const float lsel = mxl + logf(sl_warp_sum((legal[0] ? expf(l[0] - mxl) : 0.0f) + (legal[1] ? expf(l[1] - mxl) : 0.0f)));
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            logp[k] = legal[k] ? l[k] - lsel : -INFINITY;
            p[k] = legal[k] ? expf(logp[k]) : 0.0f;
        }
        const float ent = -sl_warp_sum((legal[0] && p[0] > 0.0f ? p[0] * logp[0] : 0.0f) + (legal[1] && p[1] > 0.0f ? p[1] * logp[1] : 0.0f));
        const float ill = sl_warp_sum((in[0] && !legal[0] ? q[0] : 0.0f) + (in[1] && !legal[1] ? q[1] : 0.0f));
        const float lab_logq = __shfl_sync(0xffffffffu, label >= 32 ? l[1] - lse : l[0] - lse, label & 31);
        // argmax of the probabilities, lowest index on ties
        float best = q[0];
        int arg = lane;
        if (in[1] && q[1] > best) { best = q[1]; arg = lane + 32; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
            if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
        }
        if (a.dlogits) {
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int j = lane + 32 * k;
                if (!in[k]) continue;
                float d = (q[k] - (j == label ? 1.0f : 0.0f)) * inv38B;
                if (legal[k] && p[k] > 0.0f) d += a.ent_coef * invB * p[k] * (logp[k] + ent);
                a.dlogits[b * BRL_NUM_ACTIONS + j] = d;
                sl_split_store(a, b * 64 + j, d);
            }
            if (lane >= 6) sl_split_store(a, b * 64 + 32 + lane, 0.0f);  // the value column (38) and the padding 39..63
        }
        if (lane == 0) {
            if (a.dlogits) a.dvalue[b] = 0.0f;
            s_target -= (double)lab_logq;
            s_ent += (double)ent;
            s_correct += arg == label ? 1.0 : 0.0;
            s_ill += (double)ill;
        }
    }
    // block sums, then the last block to arrive forms the statistics (k_ppo_loss's ticket)
    __shared__ double part[4][4];
    __shared__ bool last_block;
    const int w = threadIdx.x >> 5;
    if (lane == 0) { part[w][0] = s_target; part[w][1] = s_ent; part[w][2] = s_correct; part[w][3] = s_ill; }
    __syncthreads();
    if (threadIdx.x < 4) {
        const int k = threadIdx.x;
        atomicAdd(&a.acc[k], part[0][k] + part[1][k] + part[2][k] + part[3][k]);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long t = atomicAdd(reinterpret_cast<unsigned long long*>(&a.acc[kSlAccTicket]), 1ull);
        last_block = t == (unsigned long long)gridDim.x - 1ull;
    }
    __syncthreads();
    if (last_block && threadIdx.x == 0) {
        __threadfence();
        sl_finalize(a);
    }
}

struct SlHead {
    const uint8_t* mask;
    const int32_t* label;
    float* stats;
    double* acc;
    int64_t B;
    float ent_coef;
    bool backward;
};

static int32_t sl_loss_head(cudaStream_t s, const TrainHeadIO& io, const void* ctx) {
    const SlHead& h = *static_cast<const SlHead*>(ctx);
    SlLossArgs a{};
    a.logits = io.logits;
    a.mask = h.mask;
    a.label = h.label;
    if (h.backward) {
        a.dlogits = io.dlogits;
        a.dvalue = io.dvalue;
        a.dz_hi = static_cast<unsigned short*>(io.dz_hi);
        a.dz_lo = static_cast<unsigned short*>(io.dz_lo);
    }
    a.stats = h.stats;
    a.acc = h.acc;
    a.B = h.B;
    a.ent_coef = h.ent_coef;
    unsigned grid = (unsigned)((h.B + 3) / 4);
    if (grid > 148u * 8u) grid = 148u * 8u;
    launch_pdl(k_sl_loss, dim3(grid), dim3(128), 0, s, a);
    return check_launch(h.backward ? "brl_sl_grad (loss head)" : "brl_sl_eval (loss head)");
}

// brl_sl_grad: [0] obs [1] blob [2] scratch [3] mask [4] label [5] grads [6] stats [7] acc
// brl_sl_eval: [0] obs [1] blob [2] scratch [3] mask [4] label [5] stats [6] acc
static int32_t sl_minibatch(const char* what, cudaStream_t s, void** b, const void* opaque, size_t len, bool backward) {
    if (opaque == nullptr || len != sizeof(BrlSlParams))
        return fail(BRL_E_OPAQUE, "%s: opaque must be one BrlSlParams (%zu bytes), got %zu", what, sizeof(BrlSlParams), len);
    const BrlSlParams* p = static_cast<const BrlSlParams*>(opaque);
    if (p->batch < 0 || p->batch > (1 << 24)) return fail(BRL_E_OPAQUE, "%s: batch must be in [0, 2^24]", what);
    if (p->batch == 0) return BRL_OK;
    static const char* grad_names[] = {"obs", "blob", "scratch", "mask", "label", "grads", "stats", "acc"};
    static const char* eval_names[] = {"obs", "blob", "scratch", "mask", "label", "stats", "acc"};
    // obs, blob, scratch, grads and acc 16-byte aligned
    const int32_t rc = backward ? check_buffers(what, b, grad_names, 8, 0, 1u << 0 | 1u << 1 | 1u << 2 | 1u << 5 | 1u << 7)
                                : check_buffers(what, b, eval_names, 7, 0, 1u << 0 | 1u << 1 | 1u << 2 | 1u << 6);
    if (rc != BRL_OK) return rc;
    SlHead head{};
    head.mask = static_cast<const uint8_t*>(b[3]);
    head.label = static_cast<const int32_t*>(b[4]);
    head.stats = static_cast<float*>(b[backward ? 6 : 5]);
    head.acc = static_cast<double*>(b[backward ? 7 : 6]);
    head.B = p->batch;
    head.ent_coef = p->ent_coef;
    head.backward = backward;
    TrainMinibatch t{};
    t.obs = b[0];
    t.obs_flags = p->flags & (BRL_F_OBS_U8 | BRL_F_OBS_BF16);  // same bits as BRL_PPO_OBS_U8 / BRL_PPO_OBS_BF16
    t.batch = p->batch;
    t.blob = static_cast<const unsigned char*>(b[1]);
    t.scratch = static_cast<unsigned char*>(b[2]);
    t.grads = backward ? static_cast<float*>(b[5]) : nullptr;
    t.grad_sumsq = backward ? head.acc + kSlAccSumsq : nullptr;
    t.zero = head.acc;
    t.zero_bytes = 16 * sizeof(double);
    t.what = what;
    t.loss_head = sl_loss_head;
    t.ctx = &head;
    return launch_train_minibatch(s, t);
}

}  // namespace brl

using namespace brl;

extern "C" {

int32_t brl_sl_grad(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return sl_minibatch("brl_sl_grad", (cudaStream_t)stream, b, opaque, len, true);
}

int32_t brl_sl_eval(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return sl_minibatch("brl_sl_eval", (cudaStream_t)stream, b, opaque, len, false);
}

}  // extern "C"
