// brl_ppo.cu -- the PPO update's non-GEMM arithmetic (SURVEY 8f-1, src/update.py:74-242,
// ppo.py:195-211): the clipped-surrogate / clipped-value / entropy loss head fused with its
// own backward (d loss / d logits, d loss / d value in one pass over the minibatch), and the
// optimizer step (optax.clip_by_global_norm + optax.adam) over a flat parameter buffer.
// The MLP forward/backward GEMMs between them are plain library GEMMs (cuBLAS via torch).
#include "common.h"
#include "loss_head.cuh"
#include "ppo_gram.cuh"

namespace brl {

constexpr int kA = 38;

struct PpoArgs {
    const float* logits;       // [B, 38]
    const float* value;        // [B]
    const int32_t* index;      // [B] rows of the flat trajectory (NULL = identity)
    const uint8_t* mask;       // [total, 38]
    const int32_t* action;     // [total]
    const float* old_log_prob; // [total]
    const float* old_value;    // [total]
    const float* adv;          // [total]
    const float* targets;      // [total]
    float* dlogits;            // [B, 38]
    float* dvalue;             // [B]
    float* stats;              // [8]
    double* acc;               // [16] scratch accumulators; the rest of the BRL_PPO_SCRATCH_BYTES scratch follows:
    double* spec;              // [40] {sigma_max, v[38], 0} of the illegal-probability matrix (k_ppo_illegal_gram)
    float* gram_part;          // [kGramBlocks][38 * 38] per-block partial Gram matrices
    int defer_illegal;         // the statistic is formed later (a spare block of k_bias_grad); only valid with ill_coef == 0
    int skip_illegal;          // ... or not at all (BRL_PPO_ILLEGAL_STAT clear): stats[6] = NaN
    // optional (brl_ppo_grad): d loss / d (logits, value) also as bf16 hi / lo rows [B, 64] (38 logits, value, zeros),
    // the A operand of the head's input-gradient GEMM and the B operand of its weight-gradient GEMM
    unsigned short* dz_hi;
    unsigned short* dz_lo;
    int64_t B;
    float clip_eps, ent_coef, vf_coef, ill_coef;
    int value_clipping, reward_scaling, masked_policy;
};

// acc slots
enum { kAccAdv = 0, kAccAdv2, kAccIll, kAccActor, kAccValue, kAccEnt, kAccKl, kAccClip, kAccAnchorKl, kAccGramTicket = 13, kAccTicket = 15 };
static_assert(128 + 40 * 8 <= 512 && 512 + kGramBlocks * kGramN * 4 <= BRL_PPO_SCRATCH_BYTES, "scratch layout");
static_assert(kAccGramTicket == 13, "gram_args_at (ppo_gram.cuh) places the Gram ticket in f64 13");

// one warp per sample; lane owns actions lane and lane + 32
struct Row {
    float l[2];
    bool in[2], legal[2];
    __device__ __forceinline__ void load(const PpoArgs& a, int64_t b, int64_t src, int lane) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            int j = lane + 32 * k;
            in[k] = j < kA;
            l[k] = in[k] ? a.logits[b * kA + j] : -INFINITY;
            legal[k] = in[k] && a.mask[src * kA + j] != 0;
        }
    }
    __device__ __forceinline__ float softmax(const bool sel[2], float p[2], float logp[2]) const { return softmax_sel(l, sel, p, logp); }
};

// ---- the loss head of K learners at once (brl_ppo_grad_grouped): blockIdx.y = learner --------------------------------
// `a` holds learner 0's scratch pointers and the shared flags; learner k's trajectory comes from row k of the device
// table, its coefficients from row k of `coefs`, and its minibatch scratch / accumulators lie k strides further.
struct PpoGroupArgs {
    PpoArgs a;
    const long long* traj;   // [K][8]: obs, index, mask, action, old_log_prob, old_value, advantages, targets
    const float* coefs;      // [K][4]: clip_eps, ent_coef, vf_coef, illegal_l2_coef
    long long sc_stride;     // bytes between learners' minibatch scratch (logits, value, dlogits, dvalue, dz)
    long long acc_stride;    // bytes between learners' accumulator scratch
    int illegal_stat;        // BRL_PPO_ILLEGAL_STAT
};
__device__ __forceinline__ PpoArgs learner_ppo_args(const PpoGroupArgs& g, int k) {
    PpoArgs a = g.a;
    auto sc = [&](auto* p) { return (decltype(p))((const char*)p + k * g.sc_stride); };
    const long long* t = g.traj + 8 * k;
    a.logits = sc(a.logits);
    a.value = sc(a.value);
    a.dlogits = sc(a.dlogits);
    a.dvalue = sc(a.dvalue);
    a.dz_hi = sc(a.dz_hi);
    a.dz_lo = sc(a.dz_lo);
    a.index = reinterpret_cast<const int32_t*>(t[1]);
    a.mask = reinterpret_cast<const uint8_t*>(t[2]);
    a.action = reinterpret_cast<const int32_t*>(t[3]);
    a.old_log_prob = reinterpret_cast<const float*>(t[4]);
    a.old_value = reinterpret_cast<const float*>(t[5]);
    a.adv = reinterpret_cast<const float*>(t[6]);
    a.targets = reinterpret_cast<const float*>(t[7]);
    a.stats += 8 * k;
    a.acc = reinterpret_cast<double*>(reinterpret_cast<char*>(a.acc) + k * g.acc_stride);
    a.spec = reinterpret_cast<double*>(reinterpret_cast<char*>(a.acc) + 128);
    a.gram_part = reinterpret_cast<float*>(reinterpret_cast<char*>(a.acc) + 512);
    a.clip_eps = g.coefs[4 * k];
    a.ent_coef = g.coefs[4 * k + 1];
    a.vf_coef = g.coefs[4 * k + 2];
    a.ill_coef = g.coefs[4 * k + 3];
    // as brl_ppo_grad: with a zero coefficient the norm is only a statistic, formed (if asked for) beside the bias sums
    a.defer_illegal = a.ill_coef == 0.0f;
    a.skip_illegal = a.defer_illegal && !g.illegal_stat;
    return a;
}
__device__ __forceinline__ const PpoArgs& learner_args(const PpoArgs& a) { return a; }
__device__ __forceinline__ PpoArgs learner_args(const PpoGroupArgs& g) { return learner_ppo_args(g, blockIdx.y); }

// sum over the minibatch of advantages and advantages^2 (reward scaling, src/update.py:35-36)
template <class Args>  // PpoArgs, or PpoGroupArgs (blockIdx.y = learner)
__global__ void __launch_bounds__(128) k_ppo_prepass(const Args g) {
    const PpoArgs& a = learner_args(g);
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    double s_adv = 0.0, s_adv2 = 0.0;
    for (int64_t b = warp * 32 + lane; b < a.B; b += nw * 32) {
        const double g = (double)a.adv[a.index ? a.index[b] : b];
        s_adv += g;
        s_adv2 += g * g;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s_adv += __shfl_xor_sync(0xffffffffu, s_adv, o);
        s_adv2 += __shfl_xor_sync(0xffffffffu, s_adv2, o);
    }
    if (lane == 0) {
        atomicAdd(&a.acc[kAccAdv], s_adv);
        atomicAdd(&a.acc[kAccAdv2], s_adv2);
    }
}

// illegal_action_loss as the spectral norm (ppo_gram.cuh): partials + tail before the loss kernel, which then has sigma_1 / v_1
// for the statistic and the gradient
__global__ void __launch_bounds__(1024) k_ppo_illegal_gram(const GramArgs g) {
    __shared__ GramSmem sm;
    pdl_trigger();
    pdl_wait();
    gram_block<1024>(g, (int)blockIdx.x, (int)gridDim.x, sm);
}
// the partial Gram matrices only (deferred statistic: the tail runs in a spare block of k_bias_grad)
__global__ void __launch_bounds__(1024) k_ppo_gram_partial(const GramArgs g) {
    __shared__ float X[64 * kGramPad];
    pdl_trigger();
    pdl_wait();
    gram_partial<1024>(g, (int)blockIdx.x, (int)gridDim.x, X);
}

// stats = {total_loss, value_loss, loss_actor, entropy, approx_kl, clipfracs, illegal_action_loss, 0}
// (the aux tuple of _loss_fn, src/update.py:144-162); run by the last block of k_ppo_loss
__device__ __forceinline__ void ppo_finalize(const PpoArgs& a) {
    const volatile double* acc = a.acc;
    const double B = (double)a.B;
    const float value_loss = (float)(acc[kAccValue] / B), loss_actor = (float)(acc[kAccActor] / B);
    const float entropy = (float)(acc[kAccEnt] / B), ill = a.defer_illegal ? 0.0f : 0.5f * (float)((const volatile double*)a.spec)[0];
    a.stats[0] = loss_actor + a.vf_coef * value_loss - a.ent_coef * entropy + a.ill_coef * ill;
    a.stats[1] = value_loss;
    a.stats[2] = loss_actor;
    a.stats[3] = entropy;
    a.stats[4] = (float)(acc[kAccKl] / B);
    a.stats[5] = (float)(acc[kAccClip] / B);
    if (a.skip_illegal) a.stats[6] = __int_as_float(0x7fc00000);  // NaN: not computed, never a stale or wrong number
    else if (!a.defer_illegal) a.stats[6] = ill;
    a.stats[7] = 0.0f;
}
// ... and with an anchor: stats[7] = mean_b KL_b, and its term in the total
__device__ __forceinline__ void ppo_finalize_anchor(const PpoArgs& a, float kl_coef) {
    const float kl = (float)(((const volatile double*)a.acc)[kAccAnchorKl] / (double)a.B);
    a.stats[0] += kl_coef * kl;
    a.stats[7] = kl;
}

// The fixed reference policy of the KL term (k_ppo_loss<Args, PpoAnchor>): f32 anchor logits [total, 38] in the rows of the
// flat trajectory, and the coefficient as a device scalar.  A group's learner k reads table[k] and coef[k].
__device__ __forceinline__ PpoAnchor anchor_arg(const PpoAnchor& an) { return an; }
template <class... Anchor>
constexpr bool kAnchored = sizeof...(Anchor) != 0;  // (a namespace-scope constant: a local one perturbs the plain kernel's code)

// Anchor = (nothing), or PpoAnchor: the anchored instantiation (brl_ppo_grad_anchored) adds coef * mean_b KL(pi(.|s_b) ||
// alpha(.|s_b)), alpha = the anchor's softmax over the policy's own action set (the legal actions, or all 38 with
// BRL_PPO_UNMASKED_POLICY): d / d logit_j = coef / B * pi_j (log pi_j - log alpha_j - KL_b) on the set, 0 elsewhere, with
// 0 log 0 := 0.  The plain instantiation keeps the parameter list (Args, int) and compiles to the code it had before.
template <class Args, class... Anchor>  // PpoArgs, or PpoGroupArgs (blockIdx.y = learner)
__global__ void __launch_bounds__(128) k_ppo_loss(const Args g, int have_prepass, Anchor... an) {
    pdl_trigger();
    pdl_wait();
    const PpoArgs& a = learner_args(g);
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float invB = 1.0f / (float)a.B;
    float g_mean = 0.0f, g_istd = 1.0f;
    if (have_prepass) {
        double m = a.acc[kAccAdv] / (double)a.B;
        double var = a.acc[kAccAdv2] / (double)a.B - m * m;
        g_mean = (float)m;
        g_istd = 1.0f / ((float)sqrt(var > 0.0 ? var : 0.0) + 1e-8f);
    }
    // spectral norm of the illegal-probability matrix and its top right singular vector (k_ppo_illegal_gram)
    const float sigma = a.defer_illegal ? 0.0f : (float)a.spec[0];
    const bool ill_grad = a.ill_coef != 0.0f && sigma > 0.0f;
    float v1[2] = {0.0f, 0.0f};
    if (ill_grad) {
        v1[0] = (float)a.spec[1 + lane];
        v1[1] = lane < kA - 32 ? (float)a.spec[33 + lane] : 0.0f;
    }
    double s_actor = 0.0, s_value = 0.0, s_ent = 0.0, s_kl = 0.0, s_clip = 0.0;
    double s_akl = 0.0;  // sum of KL_b to the anchor
    const float* anchor = nullptr;
    float kl_coef = 0.0f;
    if constexpr (kAnchored<Anchor...>) {
        const PpoAnchor x = anchor_arg(an...);
        anchor = x.table ? reinterpret_cast<const float*>(x.table[blockIdx.y]) : x.logits;
        kl_coef = x.coef[x.table ? blockIdx.y : 0];
    }
    for (int64_t b = warp; b < a.B; b += nw) {
        const int64_t src = a.index ? a.index[b] : b;
        Row r;
        r.load(a, b, src, lane);
        // masked distribution: where(mask, logits, -inf) (src/update.py:12-16,132-137)
        float p[2], logp[2];
        r.softmax(r.legal, p, logp);
        // unmasked distribution (src/update.py:139; also the policy when masking is off, :20-24)
        float q[2], logq[2];
        r.softmax(r.in, q, logq);
        const int act = a.action[src];
        const float* pol_p = a.masked_policy ? p : q;
        const float* pol_logp = a.masked_policy ? logp : logq;
        float lp_a = __shfl_sync(0xffffffffu, act >= 32 ? pol_logp[1] : pol_logp[0], act & 31);
        // actor loss (src/update.py:115-131)
        float gae = a.adv[src];
        if (a.reward_scaling) gae = (gae - g_mean) * g_istd;
        const float logratio = lp_a - a.old_log_prob[src];
        const float ratio = expf(logratio);
        const float l1 = ratio * gae, l2 = fminf(fmaxf(ratio, 1.0f - a.clip_eps), 1.0f + a.clip_eps) * gae;
        const float loss_actor = -fminf(l1, l2);
        const bool inside = ratio >= 1.0f - a.clip_eps && ratio <= 1.0f + a.clip_eps;
        const float dl_dratio = (l1 < l2 || inside) ? -gae : 0.0f;  // min picks the unclipped term, or both coincide
        const float c_ratio = dl_dratio * ratio * invB;               // d mean(loss_actor) / d log_prob
        // entropy of the masked distribution (src/update.py:136-137)
        float ent = -((r.legal[0] && p[0] > 0.0f ? p[0] * logp[0] : 0.0f) + (r.legal[1] && p[1] > 0.0f ? p[1] * logp[1] : 0.0f));
        ent = warp_sum(ent);
        // illegal-action loss (src/update.py:138-142): x = unmasked probabilities of the illegal actions, t = x . v_1;
        // d (coef * sigma_1 / 2) / d logits_j = coef / 2 * (t / sigma_1) * (x_j v_j - q_j t)
        float qi[2] = {r.in[0] && !r.legal[0] ? q[0] : 0.0f, r.in[1] && !r.legal[1] ? q[1] : 0.0f};
        const float t_i = ill_grad ? warp_sum(qi[0] * v1[0] + qi[1] * v1[1]) : 0.0f;
        // KL to the anchor over the policy's action set: the anchor's log-softmax over that set, then
        // KL_b = sum_j pi_j (log pi_j - log alpha_j) and its gradient
        float kl_b = 0.0f, dkl[2] = {0.0f, 0.0f};
        if constexpr (kAnchored<Anchor...>) {
            const bool* sel = a.masked_policy ? r.legal : r.in;
            float al[2];
#pragma unroll
            for (int k = 0; k < 2; ++k) al[k] = sel[k] ? anchor[src * kA + lane + 32 * k] : -INFINITY;
            const float amx = warp_max(fmaxf(al[0], al[1]));
            const float alse = amx + logf(warp_sum((sel[0] ? expf(al[0] - amx) : 0.0f) + (sel[1] ? expf(al[1] - amx) : 0.0f)));
            float lr[2];
#pragma unroll
            for (int k = 0; k < 2; ++k) lr[k] = sel[k] && pol_p[k] > 0.0f ? pol_logp[k] - (al[k] - alse) : 0.0f;
            kl_b = warp_sum(pol_p[0] * lr[0] + pol_p[1] * lr[1]);
            const float c_kl = kl_coef * invB;
#pragma unroll
            for (int k = 0; k < 2; ++k) dkl[k] = sel[k] && pol_p[k] > 0.0f ? c_kl * pol_p[k] * (lr[k] - kl_b) : 0.0f;
        }
        // d total / d logits
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int j = lane + 32 * k;
            if (!r.in[k]) continue;
            float d = c_ratio * ((j == act ? 1.0f : 0.0f) - pol_p[k]);
            if (r.legal[k] && p[k] > 0.0f) d += a.ent_coef * invB * p[k] * (logp[k] + ent);  // -ent_coef * dH/dl
            if (ill_grad) d += a.ill_coef * 0.5f * (t_i / sigma) * (qi[k] * v1[k] - q[k] * t_i);
            if constexpr (kAnchored<Anchor...>) d += dkl[k];
            a.dlogits[b * kA + j] = d;
            if (a.dz_hi) store_dz(a.dz_hi, a.dz_lo, b * 64 + j, d);
        }
        if (a.dz_hi && lane >= 7) store_dz(a.dz_hi, a.dz_lo, b * 64 + 32 + lane, 0.0f);  // columns 39..63 (38 is the value, below)
        if (lane == 0) {
            // value loss (src/update.py:47-72)
            const float v = a.value[b], t = a.targets[src];
            float vl, dv;
            if (a.value_clipping) {
                const float ov = a.old_value[src];
                const float diff = v - ov;
                const float vc = ov + fminf(fmaxf(diff, -a.clip_eps), a.clip_eps);
                const float e1 = (v - t) * (v - t), e2 = (vc - t) * (vc - t);
                vl = 0.5f * fmaxf(e1, e2);
                const bool unclipped = diff >= -a.clip_eps && diff <= a.clip_eps;
                dv = (e1 > e2 || unclipped) ? (v - t) : 0.0f;  // the clipped branch is constant in v when it binds
            } else {
                vl = 0.5f * (v - t) * (v - t);
                dv = v - t;
            }
            a.dvalue[b] = a.vf_coef * dv * invB;
            if (a.dz_hi) store_dz(a.dz_hi, a.dz_lo, b * 64 + 38, a.vf_coef * dv * invB);
            s_actor += (double)loss_actor;
            s_value += (double)vl;
            s_ent += (double)ent;
            s_kl += (double)((ratio - 1.0f) - logratio);
            s_clip += fabsf(ratio - 1.0f) > a.clip_eps ? 1.0 : 0.0;
            if constexpr (kAnchored<Anchor...>) s_akl += (double)kl_b;
        }
    }
    // block-level sums first (one set of same-address f64 atomics per block, not per warp), then the last block to
    // arrive (ticket in acc[kAccTicket]) forms the statistics: no separate finalize launch.  head_block_sums (loss_head.cuh)
    // does the same for sums in acc[0..N); these go to scattered slots, and its code with a slot table would differ.
    constexpr int kSums = kAnchored<Anchor...> ? 6 : 5;  // the f64 sums: actor, value, entropy, approx KL, clip fraction (, anchor KL)
    __shared__ double part[4][kSums];
    __shared__ bool last_block;
    const int w = threadIdx.x >> 5;
    if (lane == 0) {
        part[w][0] = s_actor; part[w][1] = s_value; part[w][2] = s_ent; part[w][3] = s_kl; part[w][4] = s_clip;
        if constexpr (kAnchored<Anchor...>) part[w][5] = s_akl;
    }
    __syncthreads();
    if (threadIdx.x < kSums) {
        const int k = threadIdx.x;
        const double s = part[0][k] + part[1][k] + part[2][k] + part[3][k];
        int slot = k == 0 ? kAccActor : k == 1 ? kAccValue : k == 2 ? kAccEnt : k == 3 ? kAccKl : kAccClip;
        if constexpr (kAnchored<Anchor...>) slot = k == 5 ? kAccAnchorKl : slot;
        atomicAdd(&a.acc[slot], s);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long t = atomicAdd(reinterpret_cast<unsigned long long*>(&a.acc[kAccTicket]), 1ull);
        last_block = t == (unsigned long long)gridDim.x - 1ull;
    }
    __syncthreads();
    if (last_block && threadIdx.x == 0) {
        __threadfence();
        ppo_finalize(a);
        if constexpr (kAnchored<Anchor...>) ppo_finalize_anchor(a, kl_coef);
    }
}

// a learner with a non-zero coefficient forms its norm here in full (partials + tail: the loss gradient needs v_1), one
// with the statistic asked for only the partials, the others nothing
__global__ void __launch_bounds__(1024) k_ppo_gram_grouped(const PpoGroupArgs g) {
    __shared__ GramSmem sm;
    pdl_trigger();
    pdl_wait();
    const PpoArgs a = learner_ppo_args(g, blockIdx.y);
    if (a.skip_illegal) return;
    const GramArgs ga = gram_args_at(a.logits, a.index, a.mask, a.B, reinterpret_cast<unsigned char*>(a.acc), nullptr);
    if (a.defer_illegal) gram_partial<1024>(ga, (int)blockIdx.x, (int)gridDim.x, sm.X);
    else gram_block<1024>(ga, (int)blockIdx.x, (int)gridDim.x, sm);
}


// ---- optimizer: optax.chain(clip_by_global_norm(c), adam(lr, eps=1e-5)) (ppo.py:195-211) -------
// VEC = 4: 128-bit accesses over the first n / 4 * 4 elements (16-byte-aligned buffers), the <= 3 tail elements by block 0
template <int VEC>
__global__ void __launch_bounds__(256) k_sumsq(const float* __restrict__ g, int64_t n, double* __restrict__ out) {
    double s = 0.0;
    const int64_t n_items = n / VEC;
    if (VEC == 4 && blockIdx.x == 0 && n_items * VEC + threadIdx.x < n) {
        const double v = (double)g[n_items * VEC + threadIdx.x];
        s += v * v;
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += (int64_t)gridDim.x * blockDim.x) {
        if (VEC == 4) {
            const float4 v = reinterpret_cast<const float4*>(g)[i];
            s += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
        } else {
            const double v = (double)g[i];
            s += v * v;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ double sh[8];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < (int)(blockDim.x >> 5); ++k) t += sh[k];
        atomicAdd(out, t);
    }
}

__device__ __forceinline__ void adam_one(float& p, float g, float& m, float& v, float scale, float lr, float b1, float b2, float eps,
                                         float bc1, float bc2) {
    const float gi = g * scale;
    const float mi = b1 * m + (1.0f - b1) * gi;
    const float vi = b2 * v + (1.0f - b2) * gi * gi;
    m = mi;
    v = vi;
    p = p - lr * (mi / bc1) / (sqrtf(vi / bc2) + eps);
}

template <int VEC>
__global__ void __launch_bounds__(256) k_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                              float* __restrict__ v, int64_t n, const double* __restrict__ sumsq,
                                              float max_norm, float lr, float b1, float b2, float eps, float bc1, float bc2) {
    // optax.clip_by_global_norm: g * (max_norm / norm) only when norm >= max_norm
    float scale = 1.0f;
    if (max_norm > 0.0f) {
        const float norm = (float)sqrt(*sumsq);
        if (!(norm < max_norm)) scale = max_norm / norm;
    }
    const int64_t n_items = n / VEC;
    if (VEC == 4 && blockIdx.x == 0 && n_items * VEC + threadIdx.x < n) {
        const int64_t i = n_items * VEC + threadIdx.x;
        adam_one(p[i], g[i], m[i], v[i], scale, lr, b1, b2, eps, bc1, bc2);
    }
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += (int64_t)gridDim.x * blockDim.x) {
        if (VEC == 4) {
            float4 pi = reinterpret_cast<float4*>(p)[i], mi = reinterpret_cast<float4*>(m)[i], vi = reinterpret_cast<float4*>(v)[i];
            const float4 gi = reinterpret_cast<const float4*>(g)[i];
            adam_one(pi.x, gi.x, mi.x, vi.x, scale, lr, b1, b2, eps, bc1, bc2);
            adam_one(pi.y, gi.y, mi.y, vi.y, scale, lr, b1, b2, eps, bc1, bc2);
            adam_one(pi.z, gi.z, mi.z, vi.z, scale, lr, b1, b2, eps, bc1, bc2);
            adam_one(pi.w, gi.w, mi.w, vi.w, scale, lr, b1, b2, eps, bc1, bc2);
            reinterpret_cast<float4*>(p)[i] = pi;
            reinterpret_cast<float4*>(m)[i] = mi;
            reinterpret_cast<float4*>(v)[i] = vi;
        } else {
            adam_one(p[i], g[i], m[i], v[i], scale, lr, b1, b2, eps, bc1, bc2);
        }
    }
}

// rows of a [total, width] matrix selected by index -> [B, width] (minibatch of src/update.py:188-206)
template <class T>
__global__ void __launch_bounds__(256) k_gather_rows(const T* __restrict__ src, const int32_t* __restrict__ index,
                                                     T* __restrict__ dst, int64_t B, int width_vec) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * width_vec) return;
    const int64_t b = i / width_vec;
    const int c = (int)(i - b * width_vec);
    dst[b * width_vec + c] = src[(int64_t)index[b] * width_vec + c];
}

}  // namespace brl

using namespace brl;

extern "C" {

int32_t brl_ppo_loss(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    if (opaque == nullptr || len != sizeof(BrlPpoParams))
        return fail(BRL_E_OPAQUE, "brl_ppo_loss: opaque must be one BrlPpoParams (%zu bytes), got %zu", sizeof(BrlPpoParams), len);
    return brl::launch_ppo_loss((cudaStream_t)stream, b, static_cast<const BrlPpoParams*>(opaque), nullptr, nullptr, false, false);
}

}  // extern "C"

// blocks of `threads` threads that form the partial Gram matrices (2 samples per warp and chunk)
int brl::gram_blocks(int64_t B, int threads) {
    const int64_t chunk = 2 * (threads / 32), want = (B + chunk - 1) / chunk;
    return (int)(want < kGramBlocks ? want : kGramBlocks);
}

brl::GramArgs brl::gram_args(void** b, const BrlPpoParams* p, float* stat) {
    return gram_args_at(static_cast<const float*>(b[0]), static_cast<const int32_t*>(b[2]), static_cast<const uint8_t*>(b[3]),
                        p->batch, static_cast<unsigned char*>(b[12]), stat);
}

// The loss head's launches, for one learner (Args = PpoArgs, a = g) or K (PpoGroupArgs, a = g.a, one grid row per learner):
// `flags` decoded into `a`, then the advantage prepass (reward scaling), the Gram kernel (none when `gram` is NULL) and
// the loss kernel (with the KL term when `anchor` is set).
template <class Args, class GA>
static int32_t launch_ppo_chain(cudaStream_t s, const Args& g, PpoArgs& a, int32_t flags, unsigned K, void (*gram)(GA), const GA& ga,
                                const PpoAnchor* anchor, const char* what) {
    a.value_clipping = (flags & BRL_PPO_VALUE_CLIPPING) != 0;
    a.reward_scaling = (flags & BRL_PPO_REWARD_SCALING) != 0;
    a.masked_policy = (flags & BRL_PPO_UNMASKED_POLICY) == 0;
    const unsigned grid = head_grid(a.B);
    const int prepass = a.reward_scaling;
    if (prepass) k_ppo_prepass<Args><<<dim3(grid > 32u ? 32u : grid, K), 128, 0, s>>>(g);
    if (gram) {
        const dim3 gram_grid((unsigned)brl::gram_blocks(a.B, 1024), K);
        if (prepass) gram<<<gram_grid, 1024, 0, s>>>(ga);  // a plain launch may not be followed by a PDL one that skips it
        else launch_pdl(gram, gram_grid, dim3(1024), 0, s, ga);
    }
    if (anchor) launch_pdl(k_ppo_loss<Args, PpoAnchor>, dim3(grid, K), dim3(128), 0, s, g, prepass, *anchor);
    else launch_pdl(k_ppo_loss<Args>, dim3(grid, K), dim3(128), 0, s, g, prepass);
    return check_launch(what);
}

int32_t brl::launch_ppo_loss(cudaStream_t stream, void** b, const BrlPpoParams* p, void* dz_hi, void* dz_lo, bool acc_zeroed,
                             bool defer_illegal, const PpoAnchor* anchor) {
    if (p->batch <= 0) return fail(BRL_E_OPAQUE, "brl_ppo_loss: batch must be > 0");
    static const char* names[] = {"logits", "value", "index", "mask", "action", "old_log_prob", "old_value", "advantages",
                                  "targets", "dlogits", "dvalue", "stats", "scratch"};
    const int32_t rc = check_buffers("brl_ppo_loss", b, names, 13, 1u << 2, 0);
    if (rc != BRL_OK) return rc;
    if (reinterpret_cast<uintptr_t>(b[12]) & 15u) return fail(BRL_E_BUFFER, "brl_ppo_loss: scratch is not 16-byte aligned");
    PpoArgs a{};
    a.logits = static_cast<const float*>(b[0]);
    a.value = static_cast<const float*>(b[1]);
    a.index = static_cast<const int32_t*>(b[2]);
    a.mask = static_cast<const uint8_t*>(b[3]);
    a.action = static_cast<const int32_t*>(b[4]);
    a.old_log_prob = static_cast<const float*>(b[5]);
    a.old_value = static_cast<const float*>(b[6]);
    a.adv = static_cast<const float*>(b[7]);
    a.targets = static_cast<const float*>(b[8]);
    a.dlogits = static_cast<float*>(b[9]);
    a.dvalue = static_cast<float*>(b[10]);
    a.stats = static_cast<float*>(b[11]);
    a.acc = static_cast<double*>(b[12]);
    a.spec = reinterpret_cast<double*>(static_cast<unsigned char*>(b[12]) + 128);
    a.gram_part = reinterpret_cast<float*>(static_cast<unsigned char*>(b[12]) + 512);
    a.dz_hi = static_cast<unsigned short*>(dz_hi);
    a.dz_lo = static_cast<unsigned short*>(dz_lo);
    a.B = p->batch;
    a.clip_eps = p->clip_eps;
    a.ent_coef = p->ent_coef;
    a.vf_coef = p->vf_coef;
    a.ill_coef = p->illegal_l2_coef;
    a.defer_illegal = defer_illegal && a.ill_coef == 0.0f;
    a.skip_illegal = a.defer_illegal && !(p->flags & BRL_PPO_ILLEGAL_STAT);
    cudaStream_t s = (cudaStream_t)stream;
    if (!acc_zeroed && cudaMemsetAsync(a.acc, 0, 16 * sizeof(double), s) != cudaSuccess) return check_launch("brl_ppo_loss");
    const GramArgs g = a.skip_illegal ? GramArgs{} : brl::gram_args(b, p, nullptr);
    void (*gram)(GramArgs) = a.skip_illegal ? nullptr : a.defer_illegal ? k_ppo_gram_partial : k_ppo_illegal_gram;
    return launch_ppo_chain(s, a, a, p->flags, 1u, gram, g, anchor, "brl_ppo_loss");
}

extern "C" {

static int32_t adam_impl(brl_stream_t stream, void** b, const void* opaque, size_t len, bool presummed);
int32_t brl_adam_clip(brl_stream_t stream, void** b, const void* opaque, size_t len) { return adam_impl(stream, b, opaque, len, false); }
int32_t brl_adam_apply(brl_stream_t stream, void** b, const void* opaque, size_t len) { return adam_impl(stream, b, opaque, len, true); }

static int32_t adam_impl(brl_stream_t stream, void** b, const void* opaque, size_t len, bool presummed) {
    if (opaque == nullptr || len != sizeof(BrlAdamParams))
        return fail(BRL_E_OPAQUE, "brl_adam_clip: opaque must be one BrlAdamParams (%zu bytes), got %zu", sizeof(BrlAdamParams), len);
    const BrlAdamParams* p = static_cast<const BrlAdamParams*>(opaque);
    static const char* names[] = {"params", "grads", "m", "v", "scratch"};
    const int32_t rc = check_buffers("brl_adam_clip", b, names, 5, 0, 0);
    if (rc != BRL_OK) return rc;
    if (p->n <= 0 || p->step <= 0) return fail(BRL_E_OPAQUE, "brl_adam_clip: n and step (1-based) must be > 0");
    cudaStream_t s = (cudaStream_t)stream;
    double* sumsq = static_cast<double*>(b[4]);
    float* pp = static_cast<float*>(b[0]);
    const float* gg = static_cast<const float*>(b[1]);
    float* mm = static_cast<float*>(b[2]);
    float* vv = static_cast<float*>(b[3]);
    const bool aligned = ((reinterpret_cast<uintptr_t>(pp) | reinterpret_cast<uintptr_t>(gg) | reinterpret_cast<uintptr_t>(mm) |
                           reinterpret_cast<uintptr_t>(vv)) & 15u) == 0;
    const int64_t items = aligned ? (p->n + 3) / 4 : p->n;
    unsigned grid = (unsigned)((items + 255) / 256);
    if (grid > 148u * 8u) grid = 148u * 8u;
    if (!presummed && cudaMemsetAsync(sumsq, 0, sizeof(double), s) != cudaSuccess) return check_launch("brl_adam_clip");
    const float bc1 = 1.0f - powf(p->beta1, (float)p->step), bc2 = 1.0f - powf(p->beta2, (float)p->step);
    if (aligned) {
        if (!presummed) k_sumsq<4><<<grid, 256, 0, s>>>(gg, p->n, sumsq);
        k_adam<4><<<grid, 256, 0, s>>>(pp, gg, mm, vv, p->n, sumsq, p->max_grad_norm, p->lr, p->beta1, p->beta2, p->eps, bc1, bc2);
    } else {
        if (!presummed) k_sumsq<1><<<grid, 256, 0, s>>>(gg, p->n, sumsq);
        k_adam<1><<<grid, 256, 0, s>>>(pp, gg, mm, vv, p->n, sumsq, p->max_grad_norm, p->lr, p->beta1, p->beta2, p->eps, bc1, bc2);
    }
    return check_launch("brl_adam_clip");
}

int32_t brl_gather_rows(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    BRL_REQUIRE(b[0], "src");
    if (b[1] == nullptr) return fail(BRL_E_BUFFER, "brl_gather_rows: buffer 'index' is NULL");
    BRL_REQUIRE(b[2], "dst");
    const int64_t B = p->n_envs;
    const int row_bytes = p->k_steps;  // bytes per row
    if (row_bytes <= 0) return fail(BRL_E_OPAQUE, "brl_gather_rows: k_steps (row bytes) must be > 0");
    cudaStream_t s = (cudaStream_t)stream;
    if (row_bytes % 16 == 0) {
        const int w = row_bytes / 16;
        k_gather_rows<uint4><<<(unsigned)((B * w + 255) / 256), 256, 0, s>>>(static_cast<const uint4*>(b[0]), static_cast<const int32_t*>(b[1]),
                                                                              static_cast<uint4*>(b[2]), B, w);
    } else if (row_bytes % 2 == 0) {
        const int w = row_bytes / 2;
        k_gather_rows<uint16_t><<<(unsigned)((B * w + 255) / 256), 256, 0, s>>>(static_cast<const uint16_t*>(b[0]), static_cast<const int32_t*>(b[1]),
                                                                                 static_cast<uint16_t*>(b[2]), B, w);
    } else {
        k_gather_rows<uint8_t><<<(unsigned)((B * row_bytes + 255) / 256), 256, 0, s>>>(static_cast<const uint8_t*>(b[0]), static_cast<const int32_t*>(b[1]),
                                                                                       static_cast<uint8_t*>(b[2]), B, row_bytes);
    }
    return check_launch("brl_gather_rows");
}

}  // extern "C"

int32_t brl::launch_ppo_loss_grouped(cudaStream_t s, const PpoGroupIO& io) {
    PpoGroupArgs g{};
    PpoArgs& a = g.a;
    a.logits = io.head.logits;
    a.value = io.head.value;
    a.dlogits = io.head.dlogits;
    a.dvalue = io.head.dvalue;
    a.dz_hi = static_cast<unsigned short*>(io.head.dz_hi);
    a.dz_lo = static_cast<unsigned short*>(io.head.dz_lo);
    a.stats = io.stats;
    a.acc = reinterpret_cast<double*>(io.acc);
    a.B = io.batch;
    g.traj = io.traj;
    g.coefs = io.coefs;
    g.sc_stride = io.sc_stride;
    g.acc_stride = BRL_PPO_SCRATCH_BYTES;
    g.illegal_stat = (io.flags & BRL_PPO_ILLEGAL_STAT) != 0;
    // the Gram kernel runs for every learner: each decides from its own coefficient whether it has work
    return launch_ppo_chain(s, g, a, io.flags, (unsigned)io.K, k_ppo_gram_grouped, g, io.anchor, io.anchor ? "brl_ppo_grad_grouped_anchored" : "brl_ppo_grad_grouped");
}
