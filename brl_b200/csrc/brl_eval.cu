// brl_eval.cu -- full evaluation statistics (SURVEY 8f-2; src/evaluation.py:207-1032):
//   k_eval_act_log   per evaluation step: the acting team's masked argmax (src/evaluation.py:
//                    236-246, 650-671) fused with the per-env log update of `update_log_info`
//                    (:311-375 / :673-734): unmasked-softmax mass on illegal actions, step /
//                    pass counts and bid histograms per team, skipped for finished envs (:377-385);
//   k_eval_summary   end of match: `make_terminated_log` / `make_contract_log` per table
//                    (:448-563 / :839-925) and every mean of the `log_info` tuple (:575-596 /
//                    :986-1027) as ONE f64 vector of partial sums, all-reduced across ranks by
//                    the caller (still a single collective per match).
#include <math.h>

#include "common.h"

namespace brl {

constexpr int kAct = 38, kBids = 35;

struct ActLogArgs {
    const float* l_actor;   // [n, 38]
    const float* l_opp;     // [n, 38] or NULL (free-run opponent: always Pass, probs one-hot at Pass)
    const uint8_t* mask;    // [n, 38]
    const int8_t* current_player;
    const uint8_t* terminated;
    int32_t* action;        // [n]
    float* acc;             // [n, 76]
    int64_t n;
    int indicator_bids;     // non-duplicate `evaluate`: .at[a-3].set(1); duplicate: += 1
};

__global__ void __launch_bounds__(128) k_eval_act_log(const ActLogArgs a) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp; i < a.n; i += nw) {
        const int cur = a.current_player[i];
        const bool team1 = cur < 2;
        const float* l = team1 ? a.l_actor : a.l_opp;
        int act = 0;
        float illegal = 0.0f;
        if (l != nullptr) {
            float v[2];
            bool in[2], legal[2];
            float best = -INFINITY, mx = -INFINITY;
            int best_a = kAct;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int j = lane + 32 * k;
                in[k] = j < kAct;
                v[k] = in[k] ? l[i * kAct + j] : -INFINITY;
                legal[k] = in[k] && a.mask[i * kAct + j] != 0;
                if (legal[k] && v[k] > best) { best = v[k]; best_a = j; }
                mx = fmaxf(mx, v[k]);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ob = __shfl_xor_sync(0xffffffffu, best, o);
                const int oa = __shfl_xor_sync(0xffffffffu, best_a, o);
                if (ob > best || (ob == best && oa < best_a)) { best = ob; best_a = oa; }
                mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            }
            act = best_a < kAct ? best_a : 0;
            // pi = softmax(logits) WITHOUT the mask; illegal_action_prob = dot(pi.probs, ~mask)
            float e0 = in[0] ? expf(v[0] - mx) : 0.0f, e1 = in[1] ? expf(v[1] - mx) : 0.0f;
            float den = e0 + e1, num = (in[0] && !legal[0] ? e0 : 0.0f) + (in[1] && !legal[1] ? e1 : 0.0f);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                den += __shfl_xor_sync(0xffffffffu, den, o);
                num += __shfl_xor_sync(0xffffffffu, num, o);
            }
            illegal = num / den;
        }
        if (lane == 0) {
            a.action[i] = act;
            if (!a.terminated[i]) {
                float* r = a.acc + i * 76;
                const int t = team1 ? 0 : 1;
                r[t] += illegal;
                r[2 + t] += 1.0f;
                if (act == 0) r[4 + t] += 1.0f;
                if (act >= 3) {
                    float* bid = r + 6 + t * kBids + (act - 3);
                    *bid = a.indicator_bids ? 1.0f : *bid + 1.0f;
                }
            }
        }
    }
}

struct TableView {
    const int32_t* last_bid;
    const int32_t* last_bidder;
    const uint8_t* call_x;
    const uint8_t* call_xx;
    const float* rewards;      // [n, 4] (duplicate) or NULL
    const int32_t* pass_num;   // non-duplicate: pass-out needs _pass_num == 4 (src/evaluation.py:449-452)
};

struct SummaryArgs {
    const float* acc;           // [n, 76]
    const float* cum_return;    // [n]
    const int32_t* step_count;  // [n] state._step_count
    TableView ta, tb;           // tb.last_bid == NULL: single table (non-duplicate evaluate)
    double* sums;               // [kEvalSums]
    int64_t n;
};

// layout of the partial-sum vector
enum {
    kSN = 0, kSCum, kSCum2, kSWin, kSIllA, kSIllO, kSSteps, kSPassA, kSPassO, kSScoreA, kSScoreB,
    kSTable = 11,            // per table (9): pass_out, a_x, a_xx, o_x, o_xx, a_make, o_make, a_down, o_down
    kSBids = 29,             // actor_bid[35], opp_bid[35]
    kSContracts = 99,        // table A actor[35], opp[35]; table B actor[35], opp[35]
    kEvalSums = 239
};

__global__ void __launch_bounds__(256) k_eval_summary(const SummaryArgs a) {
    __shared__ double sh[kEvalSums];
    for (int k = threadIdx.x; k < kEvalSums; k += blockDim.x) sh[k] = 0.0;
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < a.n; i += (int64_t)gridDim.x * blockDim.x) {
        const float* r = a.acc + i * 76;
        const double cum = (double)a.cum_return[i];
        atomicAdd(&sh[kSN], 1.0);
        atomicAdd(&sh[kSCum], cum);
        atomicAdd(&sh[kSCum2], cum * cum);
        if (cum > 0.0) atomicAdd(&sh[kSWin], 1.0);
        // per-env ratios are formed in fp32 like the reference (x / y under vmap); 0/0 = NaN propagates
        atomicAdd(&sh[kSIllA], (double)(r[0] / r[2]));
        atomicAdd(&sh[kSIllO], (double)(r[1] / r[3]));
        atomicAdd(&sh[kSPassA], (double)(r[4] / r[2]));
        atomicAdd(&sh[kSPassO], (double)(r[5] / r[3]));
        atomicAdd(&sh[kSSteps], (double)a.step_count[i]);
        for (int k = 0; k < 2 * kBids; ++k)
            if (r[6 + k] != 0.0f) atomicAdd(&sh[kSBids + k], (double)r[6 + k]);
        for (int t = 0; t < 2; ++t) {
            const TableView& tv = t ? a.tb : a.ta;
            if (tv.last_bid == nullptr) continue;
            const int lb = tv.last_bid[i], who = tv.last_bidder[i];
            double* ts = sh + kSTable + 9 * t;
            if (tv.rewards) atomicAdd(&sh[t ? kSScoreB : kSScoreA], (double)tv.rewards[4 * i]);
            const bool pass_out = lb == -1 && who == -1 && (tv.pass_num == nullptr || tv.pass_num[i] == 4);
            if (pass_out) { atomicAdd(&ts[0], 1.0); continue; }
            const bool actor = who < 2;
            // NOTE the reference indexes `.at[last_bid]` even when last_bid == -1 but the env is not a
            // pass-out (cannot happen for a finished auction); guard the histogram index anyway
            if (lb >= 0 && lb < kBids) atomicAdd(&sh[kSContracts + 70 * t + (actor ? 0 : kBids) + lb], 1.0);
            if (tv.call_x[i]) atomicAdd(&ts[actor ? 1 : 3], 1.0);
            if (tv.call_xx[i]) atomicAdd(&ts[actor ? 2 : 4], 1.0);
            const float sign_src = tv.rewards ? tv.rewards[4 * i] : a.cum_return[i];
            const bool made = sign_src >= 0.0f;   // table_info.rewards[0] >= 0 / cum_return >= 0
            atomicAdd(&ts[made ? (actor ? 5 : 6) : (actor ? 7 : 8)], 1.0);
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < kEvalSums; k += blockDim.x)
        if (sh[k] != 0.0) atomicAdd(&a.sums[k], sh[k]);
}

}  // namespace brl

using namespace brl;

extern "C" {

int32_t brl_eval_num_sums(void) { return kEvalSums; }

int32_t brl_eval_act_log(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    static const char* names[] = {"logits_actor", "logits_opp", "mask", "current_player", "terminated", "action", "acc"};
    for (int k = 0; k < 7; ++k)
        if (b[k] == nullptr && k != 1) return fail(BRL_E_BUFFER, "brl_eval_act_log: buffer '%s' is NULL", names[k]);
    ActLogArgs a;
    a.l_actor = static_cast<const float*>(b[0]);
    a.l_opp = static_cast<const float*>(b[1]);
    a.mask = static_cast<const uint8_t*>(b[2]);
    a.current_player = static_cast<const int8_t*>(b[3]);
    a.terminated = static_cast<const uint8_t*>(b[4]);
    a.action = static_cast<int32_t*>(b[5]);
    a.acc = static_cast<float*>(b[6]);
    a.n = p->n_envs;
    a.indicator_bids = (p->flags & BRL_F_EVAL_INDICATOR_BIDS) != 0;
    unsigned grid = (unsigned)((a.n + 3) / 4);
    if (grid > 148u * 16u) grid = 148u * 16u;
    k_eval_act_log<<<grid, 128, 0, (cudaStream_t)stream>>>(a);
    return check_launch("brl_eval_act_log");
}

int32_t brl_eval_summary(brl_stream_t stream, void** b, const void* opaque, size_t len) {
    int32_t rc;
    const BrlParams* p = get_params(opaque, len, &rc);
    if (!p) return rc;
    if (p->n_envs == 0) return BRL_OK;  // an empty batch is a no-op; its buffers may be NULL (zero-size XLA / torch buffers)
    static const char* names[] = {"acc", "cum_return", "step_count", "a.last_bid", "a.last_bidder", "a.call_x", "a.call_xx"};
    for (int k = 0; k < 7; ++k)
        if (b[k] == nullptr) return fail(BRL_E_BUFFER, "brl_eval_summary: buffer '%s' is NULL", names[k]);
    if (b[15] == nullptr) return fail(BRL_E_BUFFER, "brl_eval_summary: buffer 'sums' is NULL");
    SummaryArgs a;
    a.acc = static_cast<const float*>(b[0]);
    a.cum_return = static_cast<const float*>(b[1]);
    a.step_count = static_cast<const int32_t*>(b[2]);
    a.ta = TableView{static_cast<const int32_t*>(b[3]), static_cast<const int32_t*>(b[4]), static_cast<const uint8_t*>(b[5]),
                     static_cast<const uint8_t*>(b[6]), static_cast<const float*>(b[7]), static_cast<const int32_t*>(b[8])};
    a.tb = TableView{static_cast<const int32_t*>(b[9]), static_cast<const int32_t*>(b[10]), static_cast<const uint8_t*>(b[11]),
                     static_cast<const uint8_t*>(b[12]), static_cast<const float*>(b[13]), static_cast<const int32_t*>(b[14])};
    a.sums = static_cast<double*>(b[15]);
    a.n = p->n_envs;
    unsigned grid = (unsigned)((a.n + 255) / 256);
    if (grid > 148u * 2u) grid = 148u * 2u;
    k_eval_summary<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    return check_launch("brl_eval_summary");
}

}  // extern "C"
