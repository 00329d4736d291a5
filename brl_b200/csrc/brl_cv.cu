// brl_cv.cu -- call-value policy improvement (not in the reference; DESIGN.md f17): the all-actions policy-gradient loss head
// on brl_call_values' training examples, riding on the tensor-core forward / backward of brl_mlp_train.cu as brl_sl.cu does.
//
//   brl_cv_grad      value_and_grad of the loss below for one minibatch: launch_train_minibatch with k_cv_loss as the head
//   brl_cv_eval      the same statistics without the backward
// The optimizer step is brl_mlp_adam_step (cvi.py: eps 1e-5 and global clipping, as ppo.train builds it).
#include "loss_head.cuh"

namespace brl {

// ---- loss head -----------------------------------------------------------------------------------------------------
// The per-sample statistics are summed as 2^-30 fixed point in int64 (exact, so independent of the block order: two calls
// on the same inputs, and brl_cv_grad / brl_cv_eval, give bit-equal stats); |x| <= 96 per sample and B <= 2^24 stay
// below 2^61.
enum { kCvAccGbar = 0, kCvAccEnt, kCvAccGarg, kCvAccRegret, kCvAccHit, kCvAccIllegal, kCvAccN, kCvAccTicket = 15 };  // 14: |grads|^2 (sl_params_minibatch)
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

// One warp per sample, lane owns calls lane and lane + 32 (loss_head.cuh).  Legal = isfinite(gain).
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
        const float mx = warp_max(fmaxf(l[0], l[1]));
        const float lse = mx + logf(warp_sum((in[0] ? expf(l[0] - mx) : 0.0f) + (in[1] ? expf(l[1] - mx) : 0.0f)));
#pragma unroll
        for (int k = 0; k < 2; ++k) q[k] = in[k] ? expf(l[k] - lse) : 0.0f;
        const float ill = warp_sum((in[0] && !legal[0] ? q[0] : 0.0f) + (in[1] && !legal[1] ? q[1] : 0.0f));
        if (!any) {
            if (a.dlogits) {
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const int j = lane + 32 * k;
                    if (!in[k]) continue;
                    a.dlogits[b * BRL_NUM_ACTIONS + j] = 0.0f;
                    store_dz(a.dz_hi, a.dz_lo, b * 64 + j, 0.0f);
                }
                if (lane >= 6) store_dz(a.dz_hi, a.dz_lo, b * 64 + 32 + lane, 0.0f);
                if (lane == 0) a.dvalue[b] = 0.0f;
            }
            if (lane == 0) s[kCvAccIllegal] += cv_fix(ill);
            continue;
        }
        // softmax over the legal calls
        softmax_sel(l, legal, p, logp);
        const float ent = -warp_sum((legal[0] && p[0] > 0.0f ? p[0] * logp[0] : 0.0f) + (legal[1] && p[1] > 0.0f ? p[1] * logp[1] : 0.0f));
        const float gbar = warp_sum((legal[0] ? p[0] * g[0] : 0.0f) + (legal[1] ? p[1] * g[1] : 0.0f));
        const float gmax = warp_max(fmaxf(legal[0] ? g[0] : -INFINITY, legal[1] ? g[1] : -INFINITY));
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
                store_dz(a.dz_hi, a.dz_lo, b * 64 + j, d);
            }
            if (lane >= 6) store_dz(a.dz_hi, a.dz_lo, b * 64 + 32 + lane, 0.0f);  // the value column (38) and the padding 39..63
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
    if (head_block_sums(s, a.acc, kCvAccTicket)) cv_finalize(a);
}

// brl_cv_grad: [0] obs [1] blob [2] scratch [3] gain [4] grads [5] stats [6] acc
// brl_cv_eval: [0] obs [1] blob [2] scratch [3] gain [4] stats [5] acc
static int32_t cv_loss_head(cudaStream_t s, const TrainHeadIO& io, const void* ctx) {
    const SlHeadCtx& h = *static_cast<const SlHeadCtx*>(ctx);
    CvLossArgs a{};
    a.logits = io.logits;
    a.gain = static_cast<const float*>(h.in[0]);
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
    launch_pdl(k_cv_loss, dim3(head_grid(h.B)), dim3(128), 0, s, a);
    return check_launch(h.backward ? "brl_cv_grad (loss head)" : "brl_cv_eval (loss head)");
}

static const char* const kCvInputs[] = {"gain"};
static const SlParamsHead kCvHead{1, kCvInputs, 1u << 0, BRL_CV_WIDE_FORWARD | BRL_CV_NARROW_BACKWARD, cv_loss_head};

}  // namespace brl

using namespace brl;

extern "C" {

int32_t brl_cv_grad(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return sl_params_minibatch("brl_cv_grad", true, (cudaStream_t)stream, b, opaque, len, kCvHead);
}

int32_t brl_cv_eval(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return sl_params_minibatch("brl_cv_eval", false, (cudaStream_t)stream, b, opaque, len, kCvHead);
}

}  // extern "C"
