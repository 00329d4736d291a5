// brl_cv.cu -- call-value policy improvement (not in the reference; DESIGN.md f17): the all-actions policy-gradient loss head
// on brl_call_values' training examples, riding on the tensor-core forward / backward of brl_mlp_train.cu as brl_sl.cu does.
//
//   brl_cv_grad      value_and_grad of the loss below for one minibatch: launch_train_minibatch with k_cv_loss as the head
//   brl_cv_eval      the same statistics without the backward
// The optimizer step is brl_mlp_adam_step (cvi.py: eps 1e-5 and global clipping, as ppo.train builds it).
#include <cuda_bf16.h>
#include <math.h>

#include "common.h"

namespace brl {

// ---- loss head -----------------------------------------------------------------------------------------------------
// The per-sample statistics are summed as 2^-30 fixed point in int64 (exact, so independent of the block order: two calls
// on the same inputs, and brl_cv_grad / brl_cv_eval, give bit-equal stats); |x| <= 96 per sample and B <= 2^24 stay
// below 2^61.
enum { kCvAccGbar = 0, kCvAccEnt, kCvAccGarg, kCvAccRegret, kCvAccHit, kCvAccIllegal, kCvAccN, kCvAccSumsq = 14, kCvAccTicket = 15 };
constexpr double kCvFix = 1073741824.0;  // 2^30
constexpr float kCvImpScale = 24.0f;     // J_b = gbar / 24: the IMP scale of reward_mode "par_imp"

struct CvLossArgs {
    const float* logits;  // [B, 38]
    const float* gain;    // [B, 38], NaN = illegal
    float* dlogits;       // [B, 38] or NULL (brl_cv_eval)
    float* dvalue;        // [B]
    unsigned short* dz_hi;
    unsigned short* dz_lo;
    float* stats;         // [8]
    double* acc;          // [16], zeroed by the caller; elements 0..5 hold int64 fixed-point sums
    int64_t B;
    float ent_coef;
};

__device__ __forceinline__ float cv_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float cv_warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ void cv_split_store(const CvLossArgs& a, int64_t idx, float v) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v), l = __float2bfloat16_rn(v - __bfloat162float(h));
    a.dz_hi[idx] = *reinterpret_cast<const unsigned short*>(&h);
    a.dz_lo[idx] = *reinterpret_cast<const unsigned short*>(&l);
}
__device__ __forceinline__ long long cv_fix(float v) { return __double2ll_rn((double)v * kCvFix); }

// stats = {total loss, mean gbar, mean g(argmax), mean regret of the argmax, entropy, argmax-is-best share, illegal mass, 0};
// run by the last block
__device__ __forceinline__ void cv_finalize(const CvLossArgs& a) {
    const volatile long long* acc = reinterpret_cast<const volatile long long*>(a.acc);
    const double B = (double)a.B;
    double mean[kCvAccN];
    for (int k = 0; k < kCvAccN; ++k) mean[k] = (double)acc[k] / kCvFix / B;
    a.stats[0] = (float)(-mean[kCvAccGbar] / (double)kCvImpScale - (double)a.ent_coef * mean[kCvAccEnt]);
    a.stats[1] = (float)mean[kCvAccGbar];
    a.stats[2] = (float)mean[kCvAccGarg];
    a.stats[3] = (float)mean[kCvAccRegret];
    a.stats[4] = (float)mean[kCvAccEnt];
    a.stats[5] = (float)mean[kCvAccHit];
    a.stats[6] = (float)mean[kCvAccIllegal];
    a.stats[7] = 0.0f;
}

// One warp per sample, lane owns calls lane and lane + 32 (k_sl_loss's layout).  Legal = isfinite(gain).
//   pi = softmax over the legal calls, gbar = sum pi_a g_a, H = entropy of pi
//   loss = -mean(gbar) / 24 - ent_coef * mean(H)
//   d loss / d l_j = -pi_j (g_j - gbar) / (24 B) + ent_coef * pi_j (log pi_j + H) / B (legal j), 0 otherwise; d / d value = 0
//   the argmax-logit legal call (lowest index on ties), its gain, max_a g_a minus it, whether it is a best call, and the
//   unmasked softmax mass on illegal calls.  A sample without a legal call adds 0 to every sum but the illegal mass (1).
__global__ void __launch_bounds__(128) k_cv_loss(const CvLossArgs a) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float inv24B = 1.0f / (kCvImpScale * (float)a.B), invB = 1.0f / (float)a.B;
    long long s[kCvAccN] = {0, 0, 0, 0, 0, 0};
    for (int64_t b = warp; b < a.B; b += nw) {
        float l[2], g[2], q[2], p[2], logp[2];
        bool in[2], legal[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int j = lane + 32 * k;
            in[k] = j < BRL_NUM_ACTIONS;
            l[k] = in[k] ? a.logits[b * BRL_NUM_ACTIONS + j] : -INFINITY;
            g[k] = in[k] ? a.gain[b * BRL_NUM_ACTIONS + j] : NAN;
            legal[k] = in[k] && isfinite(g[k]);
        }
        const bool any = __any_sync(0xffffffffu, legal[0] || legal[1]);
        // unmasked softmax: the illegal mass
        const float mx = cv_warp_max(fmaxf(l[0], l[1]));
        const float lse = mx + logf(cv_warp_sum((in[0] ? expf(l[0] - mx) : 0.0f) + (in[1] ? expf(l[1] - mx) : 0.0f)));
#pragma unroll
        for (int k = 0; k < 2; ++k) q[k] = in[k] ? expf(l[k] - lse) : 0.0f;
        const float ill = cv_warp_sum((in[0] && !legal[0] ? q[0] : 0.0f) + (in[1] && !legal[1] ? q[1] : 0.0f));
        if (!any) {
            if (a.dlogits) {
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const int j = lane + 32 * k;
                    if (!in[k]) continue;
                    a.dlogits[b * BRL_NUM_ACTIONS + j] = 0.0f;
                    cv_split_store(a, b * 64 + j, 0.0f);
                }
                if (lane >= 6) cv_split_store(a, b * 64 + 32 + lane, 0.0f);
                if (lane == 0) a.dvalue[b] = 0.0f;
            }
            if (lane == 0) s[kCvAccIllegal] += cv_fix(ill);
            continue;
        }
        // softmax over the legal calls
        const float mxl = cv_warp_max(fmaxf(legal[0] ? l[0] : -INFINITY, legal[1] ? l[1] : -INFINITY));
        const float lsel = mxl + logf(cv_warp_sum((legal[0] ? expf(l[0] - mxl) : 0.0f) + (legal[1] ? expf(l[1] - mxl) : 0.0f)));
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            logp[k] = legal[k] ? l[k] - lsel : -INFINITY;
            p[k] = legal[k] ? expf(logp[k]) : 0.0f;
        }
        const float ent = -cv_warp_sum((legal[0] && p[0] > 0.0f ? p[0] * logp[0] : 0.0f) + (legal[1] && p[1] > 0.0f ? p[1] * logp[1] : 0.0f));
        const float gbar = cv_warp_sum((legal[0] ? p[0] * g[0] : 0.0f) + (legal[1] ? p[1] * g[1] : 0.0f));
        const float gmax = cv_warp_max(fmaxf(legal[0] ? g[0] : -INFINITY, legal[1] ? g[1] : -INFINITY));
        // argmax of the legal logits, lowest index on ties
        float best = legal[0] ? l[0] : -INFINITY, bg = g[0];
        int arg = legal[0] ? lane : 64;
        if (legal[1] && (l[1] > best || arg == 64)) { best = l[1]; bg = g[1]; arg = lane + 32; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o), og = __shfl_xor_sync(0xffffffffu, bg, o);
            const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
            if (oa != 64 && (arg == 64 || ob > best || (ob == best && oa < arg))) { best = ob; bg = og; arg = oa; }
        }
        if (a.dlogits) {
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int j = lane + 32 * k;
                if (!in[k]) continue;
                float d = 0.0f;
                if (legal[k]) {
                    d = -p[k] * (g[k] - gbar) * inv24B;
                    if (p[k] > 0.0f) d += a.ent_coef * invB * p[k] * (logp[k] + ent);
                }
                a.dlogits[b * BRL_NUM_ACTIONS + j] = d;
                cv_split_store(a, b * 64 + j, d);
            }
            if (lane >= 6) cv_split_store(a, b * 64 + 32 + lane, 0.0f);  // the value column (38) and the padding 39..63
        }
        if (lane == 0) {
            if (a.dlogits) a.dvalue[b] = 0.0f;
            s[kCvAccGbar] += cv_fix(gbar);
            s[kCvAccEnt] += cv_fix(ent);
            s[kCvAccGarg] += cv_fix(bg);
            s[kCvAccRegret] += cv_fix(gmax - bg);
            s[kCvAccHit] += bg == gmax ? (long long)kCvFix : 0ll;
            s[kCvAccIllegal] += cv_fix(ill);
        }
    }
    // block sums, then the last block to arrive forms the statistics (k_sl_loss's ticket)
    __shared__ long long part[4][kCvAccN];
    __shared__ bool last_block;
    const int w = threadIdx.x >> 5;
    if (lane == 0)
        for (int k = 0; k < kCvAccN; ++k) part[w][k] = s[k];
    __syncthreads();
    if (threadIdx.x < kCvAccN) {
        const int k = threadIdx.x;
        atomicAdd(reinterpret_cast<unsigned long long*>(&a.acc[k]),
                  (unsigned long long)(part[0][k] + part[1][k] + part[2][k] + part[3][k]));
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long t = atomicAdd(reinterpret_cast<unsigned long long*>(&a.acc[kCvAccTicket]), 1ull);
        last_block = t == (unsigned long long)gridDim.x - 1ull;
    }
    __syncthreads();
    if (last_block && threadIdx.x == 0) {
        __threadfence();
        cv_finalize(a);
    }
}

struct CvHead {
    const float* gain;
    float* stats;
    double* acc;
    int64_t B;
    float ent_coef;
    bool backward;
};

static int32_t cv_loss_head(cudaStream_t s, const TrainHeadIO& io, const void* ctx) {
    const CvHead& h = *static_cast<const CvHead*>(ctx);
    CvLossArgs a{};
    a.logits = io.logits;
    a.gain = h.gain;
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
    launch_pdl(k_cv_loss, dim3(grid), dim3(128), 0, s, a);
    return check_launch(h.backward ? "brl_cv_grad (loss head)" : "brl_cv_eval (loss head)");
}

// brl_cv_grad: [0] obs [1] blob [2] scratch [3] gain [4] grads [5] stats [6] acc
// brl_cv_eval: [0] obs [1] blob [2] scratch [3] gain [4] stats [5] acc
static int32_t cv_minibatch(const char* what, cudaStream_t s, void** b, const void* opaque, size_t len, bool backward) {
    if (opaque == nullptr || len != sizeof(BrlSlParams))
        return fail(BRL_E_OPAQUE, "%s: opaque must be one BrlSlParams (%zu bytes), got %zu", what, sizeof(BrlSlParams), len);
    const BrlSlParams* p = static_cast<const BrlSlParams*>(opaque);
    if (p->batch < 0 || p->batch > (1 << 24)) return fail(BRL_E_OPAQUE, "%s: batch must be in [0, 2^24]", what);
    if (p->batch == 0) return BRL_OK;
    static const char* grad_names[] = {"obs", "blob", "scratch", "gain", "grads", "stats", "acc"};
    static const char* eval_names[] = {"obs", "blob", "scratch", "gain", "stats", "acc"};
    // obs, blob, scratch, grads and acc 16-byte aligned
    const int32_t rc = backward ? check_buffers(what, b, grad_names, 7, 0, 1u << 0 | 1u << 1 | 1u << 2 | 1u << 4 | 1u << 6)
                                : check_buffers(what, b, eval_names, 6, 0, 1u << 0 | 1u << 1 | 1u << 2 | 1u << 5);
    if (rc != BRL_OK) return rc;
    if ((reinterpret_cast<uintptr_t>(b[3]) & 3u) != 0) return fail(BRL_E_BUFFER, "%s: gain is not 4-byte aligned", what);
    CvHead head{};
    head.gain = static_cast<const float*>(b[3]);
    head.stats = static_cast<float*>(b[backward ? 5 : 4]);
    head.acc = static_cast<double*>(b[backward ? 6 : 5]);
    head.B = p->batch;
    head.ent_coef = p->ent_coef;
    head.backward = backward;
    TrainMinibatch t{};
    t.obs = b[0];
    t.obs_flags = p->flags & (BRL_F_OBS_U8 | BRL_F_OBS_BF16);  // same bits as BRL_PPO_OBS_U8 / BRL_PPO_OBS_BF16
    t.tune = (p->flags & BRL_CV_WIDE_FORWARD ? 4 : 0) | (p->flags & BRL_CV_NARROW_BACKWARD ? 16 : 0);  // BrlPpoParams.reserved's bits
    t.batch = p->batch;
    t.blob = static_cast<const unsigned char*>(b[1]);
    t.scratch = static_cast<unsigned char*>(b[2]);
    t.grads = backward ? static_cast<float*>(b[4]) : nullptr;
    t.grad_sumsq = backward ? head.acc + kCvAccSumsq : nullptr;
    t.zero = head.acc;
    t.zero_bytes = 16 * sizeof(double);
    t.what = what;
    t.loss_head = cv_loss_head;
    t.ctx = &head;
    return launch_train_minibatch(s, t);
}

}  // namespace brl

using namespace brl;

extern "C" {

int32_t brl_cv_grad(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return cv_minibatch("brl_cv_grad", (cudaStream_t)stream, b, opaque, len, true);
}

int32_t brl_cv_eval(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return cv_minibatch("brl_cv_eval", (cudaStream_t)stream, b, opaque, len, false);
}

}  // extern "C"
