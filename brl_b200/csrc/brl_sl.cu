// brl_sl.cu -- supervised bidding pre-training (sl.py of the reference): the cross-entropy + masked-entropy loss head
// that rides on the tensor-core forward / backward of brl_mlp_train.cu.  (The examples, brl_sl_examples, are a tile kernel
// of brl_env.cu, next to the env kernels whose phase 2 they share.)
//
//   brl_sl_grad      value_and_grad(loss) (sl.py:169-184, 205-206) for one minibatch: launch_train_minibatch with k_sl_loss
//                    as the loss head.
//   brl_sl_eval      loss / accuracy / illegal-action probability (sl.py:169-194, 288-301) without the backward.
// The optimizer step is brl_mlp_adam_step with eps = 1e-8 and no clipping (optax.adam(learning_rate), sl.py:166).
#include "loss_head.cuh"

namespace brl {

// ---- loss head -----------------------------------------------------------------------------------------------------
enum { kSlAccTarget = 0, kSlAccEnt, kSlAccCorrect, kSlAccIllegal, kSlAccN, kSlAccTicket = 15 };  // 14: |grads|^2 (sl_params_minibatch)

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

// One warp per sample, lane owns actions lane and lane + 32 (loss_head.cuh).
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
        const float mx = warp_max(fmaxf(l[0], l[1]));
        const float lse = mx + logf(warp_sum((in[0] ? expf(l[0] - mx) : 0.0f) + (in[1] ? expf(l[1] - mx) : 0.0f)));
#pragma unroll
        for (int k = 0; k < 2; ++k) q[k] = in[k] ? expf(l[k] - lse) : 0.0f;
        // softmax over the legal calls
        softmax_sel(l, legal, p, logp);
        const float ent = -warp_sum((legal[0] && p[0] > 0.0f ? p[0] * logp[0] : 0.0f) + (legal[1] && p[1] > 0.0f ? p[1] * logp[1] : 0.0f));
        const float ill = warp_sum((in[0] && !legal[0] ? q[0] : 0.0f) + (in[1] && !legal[1] ? q[1] : 0.0f));
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
                store_dz(a.dz_hi, a.dz_lo, b * 64 + j, d);
            }
            if (lane >= 6) store_dz(a.dz_hi, a.dz_lo, b * 64 + 32 + lane, 0.0f);  // the value column (38) and the padding 39..63
        }
        if (lane == 0) {
            if (a.dlogits) a.dvalue[b] = 0.0f;
            s_target -= (double)lab_logq;
            s_ent += (double)ent;
            s_correct += arg == label ? 1.0 : 0.0;
            s_ill += (double)ill;
        }
    }
    const double s[kSlAccN] = {s_target, s_ent, s_correct, s_ill};
    if (head_block_sums(s, a.acc, kSlAccTicket)) sl_finalize(a);
}

// brl_sl_grad: [0] obs [1] blob [2] scratch [3] mask [4] label [5] grads [6] stats [7] acc
// brl_sl_eval: [0] obs [1] blob [2] scratch [3] mask [4] label [5] stats [6] acc
static int32_t sl_loss_head(cudaStream_t s, const TrainHeadIO& io, const void* ctx) {
    const SlHeadCtx& h = *static_cast<const SlHeadCtx*>(ctx);
    SlLossArgs a{};
    a.logits = io.logits;
    a.mask = static_cast<const uint8_t*>(h.in[0]);
    a.label = static_cast<const int32_t*>(h.in[1]);
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
    launch_pdl(k_sl_loss, dim3(head_grid(h.B)), dim3(128), 0, s, a);
    return check_launch(h.backward ? "brl_sl_grad (loss head)" : "brl_sl_eval (loss head)");
}

static const char* const kSlInputs[] = {"mask", "label"};
static const SlParamsHead kSlHead{2, kSlInputs, 0u, 0, sl_loss_head};

}  // namespace brl

using namespace brl;

extern "C" {

int32_t brl_sl_grad(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return sl_params_minibatch("brl_sl_grad", true, (cudaStream_t)stream, b, opaque, len, kSlHead);
}

int32_t brl_sl_eval(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    return sl_params_minibatch("brl_sl_eval", false, (cudaStream_t)stream, b, opaque, len, kSlHead);
}

}  // extern "C"
