// env_device.cuh -- per-env device logic of the bridge-bidding environment (sm_100a).
//
// One env = 20 x u32 of packed state (5 uint4 planes in HBM, plane-major so that
// thread-per-env loads/stores are perfectly coalesced 128-bit accesses):
//
//   H[0..13]  the 424 auction-history bits of the observation, already at their
//             observation bit positions (bit i of the 480-bit observation lives in
//             word i/32, bit i%32), but indexed by ABSOLUTE seat instead of by seat
//             relative to the observer.  Every observation field is a 4-bit one-hot
//             nibble over seats (wb5/utils.py:28-46), so the observation for any
//             observer is a nibble-rotate of H -- O(15 words), no history loop.
//             nibble 0 (vulnerability) and bits >= 428 (hand) are kept zero.
//   A         dealer(2) vul_ns(1) vul_ew(1) seating(8) last_bid+1(6) bidder_seat(2)
//             call_x(1) call_xx(1) pass_num(3) terminated(1) carried(1) cur_seat(2)
//   B         turn(9) step_count(9)
//   D         first-namer table for the declarer rule (bidding_phase.py:156-159):
//             bit i = pair*5+strain named; bit 10+i = which partner (seat>>1)
//   K0,K1     `_rng_key` (src/utils.py:49)
//   deal      row of the deal / double-dummy table
//
// Semantics follow the files cited in include/brl_b200.h; pgx-only conventions are
// in conventions.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "conventions.h"

namespace brl {

constexpr int kNumActions = 38;
constexpr int kObsDim = 480;
constexpr int kObsWords = 15;
constexpr int kDealRowBytes = 48;
constexpr uint64_t kAllActions = (1ull << kNumActions) - 1ull;

struct Env {
    uint32_t H[14];
    uint32_t A, B, D;
    uint32_t key_lo, key_hi, deal;
};

// ---- field accessors --------------------------------------------------------
__device__ __forceinline__ uint32_t f_dealer(const Env& e) { return e.A & 3u; }
__device__ __forceinline__ uint32_t f_vul_ns(const Env& e) { return (e.A >> 2) & 1u; }
__device__ __forceinline__ uint32_t f_vul_ew(const Env& e) { return (e.A >> 3) & 1u; }
__device__ __forceinline__ uint32_t f_seating(const Env& e) { return (e.A >> 4) & 0xFFu; }
__device__ __forceinline__ uint32_t f_player_at(const Env& e, uint32_t seat) { return (e.A >> (4 + 2 * seat)) & 3u; }
__device__ __forceinline__ uint32_t f_lb1(const Env& e) { return (e.A >> 12) & 63u; }  // last_bid + 1
__device__ __forceinline__ uint32_t f_bidder_seat(const Env& e) { return (e.A >> 18) & 3u; }
__device__ __forceinline__ uint32_t f_x(const Env& e) { return (e.A >> 20) & 1u; }
__device__ __forceinline__ uint32_t f_xx(const Env& e) { return (e.A >> 21) & 1u; }
__device__ __forceinline__ uint32_t f_pass_num(const Env& e) { return (e.A >> 22) & 7u; }
__device__ __forceinline__ uint32_t f_terminated(const Env& e) { return (e.A >> 25) & 1u; }
__device__ __forceinline__ uint32_t f_cur_seat(const Env& e) { return (e.A >> 27) & 3u; }
__device__ __forceinline__ uint32_t f_turn(const Env& e) { return e.B & 511u; }
__device__ __forceinline__ uint32_t f_step_count(const Env& e) { return (e.B >> 9) & 511u; }

constexpr uint32_t kTermBit = 1u << 25;
// `terminated` is CARRIED on a live state: set by auto_reset on the fresh episode that
// replaced a finished one (src/utils.py:49-53) and by the quad step's OR
// (src/utils.py:128).  Such a state keeps its live legal mask; the next auto-reset
// step clears both bits (src/utils.py:33-41).
constexpr uint32_t kCarriedBit = 1u << 26;

__device__ __forceinline__ uint32_t bitfield_set(uint32_t w, uint32_t pos, uint32_t width, uint32_t v) {
    uint32_t m = ((1u << width) - 1u) << pos;
    return (w & ~m) | ((v << pos) & m);
}

// ---- packed state <-> HBM (plane-major uint4) --------------------------------
__device__ __forceinline__ void load_env(const uint4* __restrict__ st, int64_t stride, int64_t i, Env& e) {
    uint4 p0 = st[i], p1 = st[stride + i], p2 = st[2 * stride + i], p3 = st[3 * stride + i], p4 = st[4 * stride + i];
    e.H[0] = p0.x; e.H[1] = p0.y; e.H[2] = p0.z; e.H[3] = p0.w;
    e.H[4] = p1.x; e.H[5] = p1.y; e.H[6] = p1.z; e.H[7] = p1.w;
    e.H[8] = p2.x; e.H[9] = p2.y; e.H[10] = p2.z; e.H[11] = p2.w;
    e.H[12] = p3.x; e.H[13] = p3.y; e.A = p3.z; e.B = p3.w;
    e.D = p4.x; e.key_lo = p4.y; e.key_hi = p4.z; e.deal = p4.w;
}

__device__ __forceinline__ void store_env(uint4* __restrict__ st, int64_t stride, int64_t i, const Env& e) {
    st[i] = make_uint4(e.H[0], e.H[1], e.H[2], e.H[3]);
    st[stride + i] = make_uint4(e.H[4], e.H[5], e.H[6], e.H[7]);
    st[2 * stride + i] = make_uint4(e.H[8], e.H[9], e.H[10], e.H[11]);
    st[3 * stride + i] = make_uint4(e.H[12], e.H[13], e.A, e.B);
    st[4 * stride + i] = make_uint4(e.D, e.key_lo, e.key_hi, e.deal);
}

// ---- Philox4x32-10 ------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

constexpr uint32_t kTagKey = 0x4B455930u;   // "KEY0"
constexpr uint32_t kTagInit = 0x494E4954u;  // "INIT"
constexpr uint32_t kTagAct = 0x41435430u;   // "ACT0"
constexpr uint32_t kTagGum = 0x47554D30u;   // "GUM0"

__device__ __forceinline__ uint64_t make_key(uint64_t seed, uint64_t g) {
    uint4 r = philox4x32(make_uint4((uint32_t)g, (uint32_t)(g >> 32), kTagKey, 0u),
                         make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    return (uint64_t)r.x | ((uint64_t)r.y << 32);
}

// ---- reset / init ---------------------------------------------------------------
__device__ __forceinline__ void env_reset(Env& e, uint32_t deal, uint32_t dealer, uint32_t vul_ns, uint32_t vul_ew,
                                          uint32_t seating8, uint64_t key) {
#pragma unroll
    for (int w = 0; w < 14; ++w) e.H[w] = 0u;
    e.A = dealer | (vul_ns << 2) | (vul_ew << 3) | (seating8 << 4) | (dealer << 27);
    e.B = 0u;
    e.D = 0u;
    e.key_lo = (uint32_t)key;
    e.key_hi = (uint32_t)(key >> 32);
    e.deal = deal;
}

// one team (ids {0,1} or {2,3}) on N/S, the other on E/W (SURVEY A.1)
__device__ __forceinline__ uint32_t seating_code_to_players(uint32_t code) {
    uint32_t t = code & 1u, b1 = (code >> 1) & 1u, b2 = (code >> 2) & 1u;
    uint32_t pn = 2u * t + b1, ps = 2u * t + (1u - b1);
    uint32_t pe = 2u * (1u - t) + b2, pw = 2u * (1u - t) + (1u - b2);
    return pn | (pe << 2) | (ps << 4) | (pw << 6);
}

// init(key): keep one half of the split in _rng_key, draw the episode from the other.
// The draw is a pure function of the key, so a rollout can compute the NEXT episode's
// draw (and prefetch its deal row) as soon as the current episode starts.
struct EpisodeDraw {
    uint32_t key_lo, key_hi, deal, bits;  // bits = philox word holding dealer / vul / seating
};

__device__ __forceinline__ EpisodeDraw draw_episode(uint32_t key_lo, uint32_t key_hi, uint32_t n_deals) {
    uint4 r = philox4x32(make_uint4(key_lo, key_hi, kTagInit, 0u), make_uint2(0x62726C5Fu, 0x62323030u));
    return EpisodeDraw{r.x, r.y, __umulhi(r.z, n_deals), r.w};
}

__device__ __forceinline__ void env_init_from_draw(Env& e, const EpisodeDraw& d) {
    env_reset(e, d.deal, d.bits & 3u, (d.bits >> 2) & 1u, (d.bits >> 3) & 1u,
              seating_code_to_players((d.bits >> 4) & 7u), (uint64_t)d.key_lo | ((uint64_t)d.key_hi << 32));
}

__device__ __forceinline__ void env_init(Env& e, uint64_t key, uint32_t n_deals) {
    env_init_from_draw(e, draw_episode((uint32_t)key, (uint32_t)(key >> 32), n_deals));
}

// src/duplicate.py:113-129: seats handed to the other team ([1,0,3,2]), same deal /
// dealer / vulnerability, everything else (rng key included) back to defaults
__device__ __forceinline__ void env_duplicate_init(Env& e) {
    uint32_t s = f_seating(e);
    uint32_t p0 = s & 3u, p1 = (s >> 2) & 3u, p2 = (s >> 4) & 3u, p3 = (s >> 6) & 3u;
    uint32_t swapped = p1 | (p0 << 2) | (p3 << 4) | (p2 << 6);
    env_reset(e, e.deal, f_dealer(e), f_vul_ns(e), f_vul_ew(e), swapped, 0ull);
}

// ---- legal actions ----------------------------------------------------------------
// bidding_phase.py:51-52,157-178.  bit a of the result = action a is legal.
__device__ __forceinline__ uint64_t env_legal_mask(const Env& e) {
#if BRL_CONV_TERMINAL_MASK_ALL_TRUE
    if (f_terminated(e) && !(e.A & kCarriedBit)) return kAllActions;
#endif
    uint32_t lb1 = f_lb1(e);
    uint64_t m = kAllActions ^ ((1ull << (lb1 + 3u)) - 1ull);  // bids above the last bid
    m |= 1ull;                                                  // Pass
    if (lb1 != 0u) {
        uint32_t partner = ((f_cur_seat(e) ^ f_bidder_seat(e)) & 1u) ^ 1u;  // same parity = same side
        uint32_t x = f_x(e), xx = f_xx(e);
        if (!x && !xx && !partner) m |= 2ull;
        if (x && !xx && partner) m |= 4ull;
    }
    return m;
}

// ---- scoring -- score.py:5-106 in closed form (checked against the full table) -------
__device__ __forceinline__ int32_t contract_score(uint32_t bid, uint32_t x, uint32_t xx, uint32_t vul, int32_t tricks) {
    int32_t level = (int32_t)(bid / 5u) + 1;
    uint32_t strain = bid % 5u;
    int32_t need = level + 6;
    if (need > tricks) {
        int32_t n = need - tricks;
        int32_t s;
        if (!x && !xx) s = (vul ? 100 : 50) * n;
        else {
            s = vul ? 300 * n - 100 : (n <= 3 ? 200 * n - 100 : 300 * n - 400);
            if (xx) s *= 2;
        }
        return -s;
    }
    int32_t over = tricks - need;
    int32_t per = strain <= 1u ? 20 : 30;
    int32_t score = per * level + (strain == 4u ? 10 : 0);
    if (xx) score *= 4; else if (x) score *= 2;
    if (score >= 100) {
        score += vul ? 450 : 250;
        if (level >= 6) {
            score += vul ? 750 : 500;
            if (level == 7) score += vul ? 750 : 500;
        }
    }
    score += 50;
    if (xx) { score += 100; per = vul ? 400 : 200; }
    else if (x) { score += 50; per = vul ? 200 : 100; }
    return score + per * over;
}

// src/duplicate.py:46-69: number of thresholds reached by |d|, signed by d >= 0
__device__ __forceinline__ float imp_of_difference(float d) {
    float ad = fabsf(d);
    int imp = 0;
    constexpr float T[24] = {20, 50, 90, 130, 170, 220, 270, 320, 370, 430, 500, 600,
                             750, 900, 1100, 1300, 1500, 1750, 2000, 2250, 2500, 3000, 3500, 4000};
#pragma unroll
    for (int k = 0; k < 24; ++k) imp += ad >= T[k];
    return d >= 0.0f ? (float)imp : -(float)imp;
}

// ---- double-dummy par (not in the reference; DESIGN.md f13, restated by tests/par_ref.py) ----------------------------
// Par is the minimax value of this game over the deal's DD table t[seat][strain]:
//   - side o (NS = seats 0/2, EW = 1/3) declaring bid c scores, with T the tricks of its declarer (the partner with more
//     tricks in the strain; on a tie the one who comes first in the auction from the dealer),
//     contract_score(c, undoubled, vul_o, T) when T >= level + 6 and contract_score(c, doubled, vul_o, T) otherwise;
//     the NS score is that value for o = NS and its negative for o = EW;
//   - the sides alternate, the dealer's side first.  With no contract the side to move passes or names any contract, and
//     two passes with no contract pass the board out (0).  When o owns c the other side passes (the game ends at c) or
//     names a contract c' > c, which makes it the owner with o to move;
//   - NS maximises and EW minimises the NS score.
// The par contract ends the line on which every side to move takes, among its best options, pass if it is one of them and
// otherwise the lowest contract.  It is -1 when passed out, else bid | declarer_seat << 8 | doubled << 10.  This is a
// definition of this project: no DDS par solver is involved, and the declarer rule is a simplification.
struct Par {
    int32_t ns;        // par in NS points
    int32_t contract;  // par contract code
};

template <class Rows>
__device__ __forceinline__ Par par_score(const Env& e, const Rows& rows) {
    const uint32_t dealer = f_dealer(e);
    int32_t tr[2][5];
    uint32_t decl[2][5];
#pragma unroll
    for (uint32_t o = 0; o < 2u; ++o) {
        const bool o_first = ((o - dealer) & 3u) < ((o + 2u - dealer) & 3u);
#pragma unroll
        for (uint32_t s = 0; s < 5u; ++s) {
            const int32_t a = rows.tricks(e.deal, o, s), b = rows.tricks(e.deal, o + 2u, s);
            const bool pick_a = a > b || (a == b && o_first);
            tr[o][s] = pick_a ? a : b;
            decl[o][s] = pick_a ? o : o + 2u;
        }
    }
    const uint32_t vul[2] = {f_vul_ns(e), f_vul_ew(e)};
    auto value = [&](uint32_t o, uint32_t c) {
        const int32_t t = tr[o][c % 5u];
        const int32_t s = contract_score(c, t < (int32_t)(c / 5u) + 7 ? 1u : 0u, 0u, vul[o], t);
        return o == 0u ? s : -s;
    };
    // backward induction: V[o][c] = the value when o owns c and the other side m is to move, the better for m of passing
    // and best[m] (m's optimum over its contracts above c)
    int32_t V[2][35];
    int32_t best[2] = {INT32_MIN, INT32_MAX};  // NS maximises, EW minimises
    for (int c = 34; c >= 0; --c) {
        const int32_t v0 = min(value(0u, (uint32_t)c), best[1]);
        const int32_t v1 = max(value(1u, (uint32_t)c), best[0]);
        V[0][c] = v0;
        V[1][c] = v1;
        best[0] = max(best[0], v0);
        best[1] = min(best[1], v1);
    }
    const uint32_t d = dealer & 1u;
    auto opt = [](uint32_t side, int32_t a, int32_t b) { return side == 0u ? max(a, b) : min(a, b); };
    const int32_t after_pass = opt(d ^ 1u, 0, best[d ^ 1u]);  // the dealer's side passed: the other side's choice
    const int32_t root = opt(d, after_pass, best[d]);
    // the par line: pass when it is among the best options, else the lowest best contract
    int owner = -1, c = -1;
    int32_t target = root;
    if (after_pass != root) owner = (int)d;
    else if (after_pass != 0) owner = (int)(d ^ 1u), target = after_pass;
    while (owner >= 0) {
        int k = c + 1;
        while (V[owner][k] != target) ++k;  // a best option exists: target is the optimum over these contracts
        c = k;
        if (value((uint32_t)owner, (uint32_t)c) == target) break;  // the other side passes
        owner ^= 1;
    }
    if (owner < 0) return Par{0, -1};
    const uint32_t strain = (uint32_t)c % 5u;
    const uint32_t doubled = tr[owner][strain] < c / 5 + 7 ? 1u : 0u;
    return Par{root, c | (int32_t)(decl[owner][strain] << 8) | (int32_t)(doubled << 10)};
}

// ---- bidding-system statistics (not in the reference; DESIGN.md f15, restated by tests/system_ref.py) --------------------
// A decision is one call a (0 Pass, 1 X, 2 XX, 3 + bid) of the player at seat s.  Its context depends only on the earlier
// calls c_0 .. c_{t-1} of the auction (call k made by seat (dealer + k) mod 4):
//   0 + t     OPEN(t)         every earlier call is Pass (t = the caller's position after the dealer)
//   4 + b     RESPONSE(b)     the only bid so far is b, made by the caller's partner at call t - 2; call t - 1 was Pass; no X / XX
//   39 + b    OVERCALL(b)     the only bid so far is b, made by the caller's right-hand opponent at call t - 1
//   74        OTHER           everything else
// The histogram hist[M, 75, 38, 96] (u32, +=) holds per net, context and call: columns 0..37 the HCP histogram, 38 + 14 suit
// + len the suit-length histograms (clubs, diamonds, hearts, spades), 94 the balanced hands (no void or singleton, at most
// one doubleton: 4333, 4432, 5332), 95 the decisions.  One call adds at most one to a cell per decision it counts.
constexpr int kSysContexts = 75;
constexpr int kSysOther = 74;
constexpr int kSysCols = 96;
constexpr int64_t kSysCells = (int64_t)kSysContexts * kNumActions * kSysCols;  // u32 per net

// what the context needs from the calls before call t
struct SystemPrefix {
    uint32_t t;       // calls so far
    uint32_t bids;    // bids so far, saturating at 2
    uint32_t bid;     // the last bid (0..34)
    uint32_t bid_at;  // its call index
    uint32_t doubled; // an X or XX so far
};

__device__ __forceinline__ uint32_t system_context(const SystemPrefix& p) {
    if (p.bids == 0u) return p.t < 4u ? p.t : (uint32_t)kSysOther;  // no bid: every earlier call is Pass
    if (p.bids > 1u || p.doubled) return (uint32_t)kSysOther;
    if (p.bid_at + 1u == p.t) return 39u + p.bid;                    // right-hand opponent's bid, the call just made
    if (p.bid_at + 2u == p.t) return 4u + p.bid;                     // partner's bid, then a Pass (no bid, no X / XX since)
    return (uint32_t)kSysOther;
}

// reader 1: the prefix from the packed state (the match loop).  The bid nibbles of the history say whether a bid below the
// last one was made; X / XX are cleared by a bid, so with one bid they are the doubles of the whole auction, and the calls
// after the last bid or double are pass_num passes.
__device__ __forceinline__ SystemPrefix system_prefix(const Env& e) {
    SystemPrefix p;
    const uint32_t lb1 = f_lb1(e);
    p.t = f_turn(e);
    p.bid = lb1 - 1u;
    p.doubled = f_x(e) | f_xx(e);
    p.bid_at = p.t - 1u - f_pass_num(e);
    uint32_t below = 0u;
#pragma unroll
    for (int b = 0; b < 35; ++b) {
        const int bit = 4 * (2 + 3 * b);  // nibble of bid b (wb5/utils.py:36-38)
        if ((uint32_t)b + 1u < lb1) below |= (e.H[bit >> 5] >> (bit & 31)) & 15u;
    }
    p.bids = lb1 == 0u ? 0u : (below ? 2u : 1u);
    return p;
}

// reader 2: the prefix of a stored call sequence, one call at a time
__device__ __forceinline__ void system_push(SystemPrefix& p, uint32_t call) {
    if (call >= 3u) {
        p.bids = p.bids < 2u ? p.bids + 1u : 2u;
        p.bid = call - 3u;
        p.bid_at = p.t;
    } else if (call != 0u) {
        p.doubled = 1u;
    }
    ++p.t;
}

// hand features of a 52-bit hand mask (card c = rank * 4 + suit, rank 0 = '2' .. 12 = 'A')
struct HandFeatures {
    uint32_t hcp, len[4], balanced;
};

__device__ __forceinline__ HandFeatures hand_features(uint64_t hand) {
    constexpr uint64_t kSuit = 0x0001111111111111ull;  // bits 0, 4, .., 48: the 13 cards of clubs
    HandFeatures f;
    uint32_t shortest = 13u, doubletons = 0u;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        f.len[s] = (uint32_t)__popcll(hand & (kSuit << s));
        shortest = min(shortest, f.len[s]);
        doubletons += f.len[s] == 2u;
    }
    f.hcp = (uint32_t)__popcll((hand >> 36) & 15u) + 2u * (uint32_t)__popcll((hand >> 40) & 15u) +
            3u * (uint32_t)__popcll((hand >> 44) & 15u) + 4u * (uint32_t)__popcll((hand >> 48) & 15u);
    f.balanced = shortest >= 2u && doubletons <= 1u;
    return f;
}

// one decision into a net's histogram (hist_m = u32[75, 38, 96])
__device__ __forceinline__ void system_count(uint32_t* __restrict__ hist_m, uint32_t context, uint32_t call, const HandFeatures& f) {
    uint32_t* row = hist_m + ((size_t)context * kNumActions + call) * kSysCols;
    atomicAdd(row + f.hcp, 1u);
#pragma unroll
    for (int s = 0; s < 4; ++s) atomicAdd(row + 38 + 14 * s + f.len[s], 1u);
    if (f.balanced) atomicAdd(row + 94, 1u);
    atomicAdd(row + 95, 1u);
}

// ---- counterfactual call values (not in the reference; DESIGN.md f16, restated by tests/call_values_ref.py) ---------------
// A decision d is a step of a duplicate match's env at table T (A or B) in state S_d: player p (net m by brl_model_rows'
// rule) makes call b_d in context c = system_context(system_prefix(S_d)).  For every call a legal in S_d the branch (d, a)
// steps S_d with a (no auto-reset, no table switch) and plays that one table to its end, every player acting with its own
// net (masked argmax); r_d(a) is the branch's final rewards[0].  With R_A, R_B the match's final rewards[0] at both tables:
//   gain g_d(a) = sigma_p * (imp_of_difference(r_d(a) + R_other) - imp_of_difference(R_A + R_B)), sigma_p = +1 for players
//   0/1 and -1 for 2/3: the change of the decider's team's match IMPs, the other table held at its result; an integer in
//   [-48, 48].  regret_d = max over legal a of g_d(a) >= 0.  The played branch is the base game, so r_d(b_d) = R_T.
constexpr int kCvStats = 4;  // {n, sum x, sum x^2, #(x > 0)}

__device__ __forceinline__ int32_t call_value_gain(float r, float r_other, float base_imp, bool team1) {
    const int32_t g = (int32_t)imp_of_difference(r + r_other) - (int32_t)base_imp;
    return team1 ? g : -g;
}

__device__ __forceinline__ void history_set_bit(Env& e, uint32_t bit) {
    uint32_t w = bit >> 5, m = 1u << (bit & 31u);
#pragma unroll
    for (int k = 0; k < 14; ++k)
        if (w == (uint32_t)k) e.H[k] |= m;
}

// ---- deal-row access ------------------------------------------------------------------
// A step needs two facts about the deal: the observer's 52-bit hand mask and, at a
// terminal, one double-dummy nibble.  TableRows gathers them from the (L2-resident)
// table on demand -- right for one-launch-per-step kernels.  CachedRow holds the
// whole 48-byte row in registers -- the rollout kernels load it once per episode and
// prefetch the NEXT episode's row (its key is known in advance), which takes both
// dependent gathers off the per-step critical path.
struct TableRows {
    const uint8_t* __restrict__ table;
    __device__ __forceinline__ int32_t tricks(uint32_t deal, uint32_t seat, uint32_t strain) const {
        uint32_t t = seat * 5u + strain;
        uint32_t byte = table[(size_t)deal * kDealRowBytes + 32u + (t >> 1)];
        return (int32_t)((t & 1u) ? (byte >> 4) : (byte & 15u));
    }
    __device__ __forceinline__ uint64_t hand(uint32_t deal, uint32_t seat) const {
        const uint2 hm = *reinterpret_cast<const uint2*>(table + (size_t)deal * kDealRowBytes + 8u * seat);
        return (uint64_t)hm.x | ((uint64_t)hm.y << 32);
    }
};

struct CachedRow {
    uint4 h01, h23, dd;  // hands N,E | hands S,W | 20 DD nibbles (80 bits) + pad
    __device__ __forceinline__ void load(const uint8_t* __restrict__ table, uint32_t deal) {
        const uint4* r = reinterpret_cast<const uint4*>(table + (size_t)deal * kDealRowBytes);
        h01 = r[0];
        h23 = r[1];
        dd = r[2];
    }
    __device__ __forceinline__ int32_t tricks(uint32_t, uint32_t seat, uint32_t strain) const {
        uint32_t t = seat * 5u + strain;  // nibble index 0..19
        uint32_t w = t < 8u ? dd.x : (t < 16u ? dd.y : dd.z);
        return (int32_t)((w >> ((t & 7u) * 4u)) & 15u);
    }
    __device__ __forceinline__ uint64_t hand(uint32_t, uint32_t seat) const {
        uint32_t lo = seat == 0u ? h01.x : (seat == 1u ? h01.z : (seat == 2u ? h23.x : h23.z));
        uint32_t hi = seat == 0u ? h01.y : (seat == 1u ? h01.w : (seat == 2u ? h23.y : h23.w));
        return (uint64_t)lo | ((uint64_t)hi << 32);
    }
};

// ---- step ---------------------------------------------------------------------------
// pgx core.Env.step around bidding_phase.py:119-180; returns rewards by player id.
template <class Rows>
__device__ __forceinline__ float4 env_step(Env& e, int32_t action, const Rows& rows,
                                           float illegal_penalty, float illegal_bonus) {
    float4 rew = make_float4(0.f, 0.f, 0.f, 0.f);
    if (f_terminated(e)) return rew;  // finished env: zero-reward no-op (src/evaluation.py:120-122)

    uint32_t seat = f_cur_seat(e);
    uint64_t legal = env_legal_mask(e);
    bool illegal = action < 0 || action >= kNumActions || !((legal >> action) & 1ull);
    e.B = bitfield_set(e.B, 9, 9, f_step_count(e) + 1u);
    if (illegal) {  // SURVEY A.6.2 (unpinned convention)
        uint32_t actor = f_player_at(e, seat);
        rew = make_float4(illegal_bonus, illegal_bonus, illegal_bonus, illegal_bonus);
        if (actor == 0u) rew.x = illegal_penalty;
        else if (actor == 1u) rew.y = illegal_penalty;
        else if (actor == 2u) rew.z = illegal_penalty;
        else rew.w = illegal_penalty;
        e.A |= kTermBit;
        return rew;
    }

    uint32_t lb1 = f_lb1(e), pass_num = f_pass_num(e);
    bool finished = false;
    uint32_t hist_nibble = 0u;  // nibble of the observation this call is recorded in (0 = not recorded)
    if (action == 0) {
        pass_num += 1u;
        finished = (pass_num == 4u) || (pass_num == 3u && lb1 != 0u);
        if (lb1 == 0u) hist_nibble = 1u;  // opening pass nibble (wb5/utils.py:39-41)
    } else if (action == 1) {
        e.A |= 1u << 20;
        pass_num = 0u;
        hist_nibble = 2u + 3u * (lb1 - 1u) + 1u;  // wb5/utils.py:42-43
    } else if (action == 2) {
        e.A |= 1u << 21;
        pass_num = 0u;
        hist_nibble = 2u + 3u * (lb1 - 1u) + 2u;  // wb5/utils.py:44-45
    } else {
        uint32_t bid = (uint32_t)action - 3u;
        lb1 = bid + 1u;
        e.A = bitfield_set(e.A, 12, 6, lb1);
        e.A = bitfield_set(e.A, 18, 2, seat);
        e.A &= ~(3u << 20);  // x = xx = 0
        pass_num = 0u;
        uint32_t i = (seat & 1u) * 5u + bid % 5u;  // bidding_phase.py:156-159
        if (!((e.D >> i) & 1u)) e.D |= (1u << i) | ((seat >> 1) << (10u + i));
        hist_nibble = 2u + 3u * bid;  // wb5/utils.py:36-38
    }
    if (hist_nibble) history_set_bit(e, 4u * hist_nibble + seat);
    e.A = bitfield_set(e.A, 22, 3, pass_num);
    e.B = bitfield_set(e.B, 0, 9, f_turn(e) + 1u);

    if (finished) {
        e.A |= kTermBit;
#if BRL_CONV_TERMINAL_ADVANCES_PLAYER
        e.A = bitfield_set(e.A, 27, 2, (seat + 1u) & 3u);
#endif
        if (lb1 != 0u) {  // bidding_phase.py:182-206, score.py:109-125, contract.py:94-106
            uint32_t bid = lb1 - 1u, strain = bid % 5u;
            uint32_t pair = f_bidder_seat(e) & 1u;
            uint32_t i = pair * 5u + strain;
            uint32_t decl_seat = pair + 2u * ((e.D >> (10u + i)) & 1u);
            uint32_t vul = pair ? f_vul_ew(e) : f_vul_ns(e);
            int32_t tricks = rows.tricks(e.deal, decl_seat, strain);
            float s = (float)contract_score(bid, f_x(e), f_xx(e), vul, tricks);
            uint32_t team = f_player_at(e, decl_seat) >> 1;
            float s01 = team == 0u ? s : -s;
            rew = make_float4(s01, s01, -s01, -s01);
        }
    } else {
        e.A = bitfield_set(e.A, 27, 2, (seat + 1u) & 3u);
    }
    return rew;
}

// src/utils.py:33-56 auto_reset around env_step; the terminal flag survives the reset
__device__ __forceinline__ float4 env_step_autoreset(Env& e, int32_t action, const uint8_t* __restrict__ table,
                                                     uint32_t n_deals, float illegal_penalty, float illegal_bonus) {
    if (f_terminated(e)) {
        e.A &= ~(kTermBit | kCarriedBit);
        e.B = bitfield_set(e.B, 9, 9, 0u);
    }
    float4 rew = env_step(e, action, TableRows{table}, illegal_penalty, illegal_bonus);
    if (f_terminated(e)) {
        env_init(e, (uint64_t)e.key_lo | ((uint64_t)e.key_hi << 32), n_deals);
        e.A |= kTermBit | kCarriedBit;
    }
    return rew;
}

// Same auto-reset step for the persistent rollout kernels: the current deal row lives in
// registers, and the next episode (draw + row) was prefetched when this one started.
struct EpisodeCache {
    CachedRow cur, next;
    EpisodeDraw next_draw;
    __device__ __forceinline__ void prime(const Env& e, const uint8_t* __restrict__ table, uint32_t n_deals) {
        cur.load(table, e.deal);
        next_draw = draw_episode(e.key_lo, e.key_hi, n_deals);
        next.load(table, next_draw.deal);
    }
};

__device__ __forceinline__ float4 env_step_autoreset_cached(Env& e, EpisodeCache& c, int32_t action,
                                                            const uint8_t* __restrict__ table, uint32_t n_deals,
                                                            float illegal_penalty, float illegal_bonus) {
    if (f_terminated(e)) {
        e.A &= ~(kTermBit | kCarriedBit);
        e.B = bitfield_set(e.B, 9, 9, 0u);
    }
    float4 rew = env_step(e, action, c.cur, illegal_penalty, illegal_bonus);
    if (f_terminated(e)) {
        env_init_from_draw(e, c.next_draw);
        e.A |= kTermBit | kCarriedBit;
        c.cur = c.next;
        c.next_draw = draw_episode(e.key_lo, e.key_hi, n_deals);
        c.next.load(table, c.next_draw.deal);  // consumed >= 4 calls from now: latency hidden
    }
    return rew;
}

// Variant for the warp-specialised rollout, where one warp runs 32 envs for many steps.
// Holding the prefetched row in REGISTERS creates a false dependency there: the warp's
// scoreboard is per register, not per lane, and some lane resets in ~96 % of the steps, so
// the reset branch of step s touches the registers that step s-1's (other lanes') row load
// is still writing -- ncu showed 31 % of the env warp's time on that long-scoreboard wait.
// Here the next episode's row is fetched with cp.async into a per-lane shared-memory slot and
// its arrival is tracked by a per-lane mbarrier, so a lane only ever waits on ITS OWN copy,
// issued at least 4 calls earlier.  Two slots per lane alternate (no WAR hazard on the slot).
struct RowSlots {  // one per lane, in shared memory (arrays indexed [slot][lane])
    uint4* rows;             // [2][EPB][3]
    unsigned long long* bar;  // [2][EPB]
    int epb;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

struct EpisodePrefetch {
    CachedRow cur;
    EpisodeDraw next_draw;
    uint32_t slot;    // slot the NEXT episode's row is arriving in
    uint32_t parity;  // bit k = phase parity to wait for on slot k's mbarrier

#ifdef BRL_PLAIN_EPISODE_LOAD
    // Debug build (scripts/racecheck_prefetch.sh): no cp.async / mbarrier at all -- the next episode's row is read with plain
    // loads when the episode starts.  Same results; compute-sanitizer racecheck then has nothing left to warn about, which
    // shows that its four warnings on the prefetch slots come from not modelling mbarrier-tracked cp.async completion.
    __device__ __forceinline__ void issue(const RowSlots&, int, const uint8_t* __restrict__) {}
#else
    __device__ __forceinline__ void issue(const RowSlots& rs, int lane, const uint8_t* __restrict__ table) {
        const uint8_t* g = table + (size_t)next_draw.deal * kDealRowBytes;
        const uint32_t dst = smem_u32(rs.rows + ((size_t)slot * rs.epb + lane) * 3);
        const uint32_t bar = smem_u32(rs.bar + (size_t)slot * rs.epb + lane);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(g) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + 16u), "l"(g + 16) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + 32u), "l"(g + 32) : "memory");
        asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
    }
#endif
    __device__ __forceinline__ void prime(const Env& e, const RowSlots& rs, int lane, const uint8_t* __restrict__ table,
                                          uint32_t n_deals) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(rs.bar + lane)) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(rs.bar + rs.epb + lane)) : "memory");
        cur.load(table, e.deal);
        next_draw = draw_episode(e.key_lo, e.key_hi, n_deals);
        slot = 0u;
        parity = 0u;
        issue(rs, lane, table);
    }
    // the episode ended: the prefetched row becomes current, start fetching the one after
    __device__ __forceinline__ void advance(const Env& e, const RowSlots& rs, int lane, const uint8_t* __restrict__ table,
                                            uint32_t n_deals) {
#ifdef BRL_PLAIN_EPISODE_LOAD
        cur.load(table, next_draw.deal);
#else
        const uint32_t bar = smem_u32(rs.bar + (size_t)slot * rs.epb + lane);
        const uint32_t want = (parity >> slot) & 1u;
        uint32_t done = 0u;
        while (!done) {
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(done) : "r"(bar), "r"(want) : "memory");
        }
        const uint4* r = rs.rows + ((size_t)slot * rs.epb + lane) * 3;
        cur.h01 = r[0];
        cur.h23 = r[1];
        cur.dd = r[2];
#endif
        parity ^= 1u << slot;
        slot ^= 1u;
        next_draw = draw_episode(e.key_lo, e.key_hi, n_deals);
        issue(rs, lane, table);
    }
};

__device__ __forceinline__ float4 env_step_autoreset_prefetch(Env& e, EpisodePrefetch& c, const RowSlots& rs, int lane,
                                                              int32_t action, const uint8_t* __restrict__ table,
                                                              uint32_t n_deals, float illegal_penalty, float illegal_bonus) {
    if (f_terminated(e)) {
        e.A &= ~(kTermBit | kCarriedBit);
        e.B = bitfield_set(e.B, 9, 9, 0u);
    }
    float4 rew = env_step(e, action, c.cur, illegal_penalty, illegal_bonus);
    if (f_terminated(e)) {
        env_init_from_draw(e, c.next_draw);
        e.A |= kTermBit | kCarriedBit;
        c.advance(e, rs, lane, table, n_deals);
    }
    return rew;
}

// ---- observation -- wb5/utils.py:15-52 as 15 words of bits ------------------------------
__device__ __forceinline__ uint32_t rotr_nibbles(uint32_t h, uint32_t q) {
    // relative seat = (absolute - observer) mod 4: rotate every nibble right by q
    uint32_t lo = 0x0F0F0F0Fu >> q;            // per-nibble mask of bits that stay after >> q
    lo = (lo & 0x0F0F0F0Fu);                   // (0xF >> q) in the low nibble of each byte
    lo |= lo << 4;
    return ((h >> q) & lo) | ((h << (4u - q)) & ~lo);
}

template <class Rows>
__device__ __forceinline__ void env_observe_words(const Env& e, const Rows& rows, uint32_t q,
                                                  uint32_t R[kObsWords]) {
#pragma unroll
    for (int w = 0; w < 14; ++w) R[w] = rotr_nibbles(e.H[w], q);
    uint32_t us = (q & 1u) ? f_vul_ew(e) : f_vul_ns(e);
    uint32_t them = (q & 1u) ? f_vul_ns(e) : f_vul_ew(e);
    R[0] |= (us ? 2u : 1u) | (them ? 8u : 4u);  // wb5/utils.py:15-16
    uint64_t hand = rows.hand(e.deal, q);
    R[13] |= (uint32_t)(hand << 12);  // observation bits 428..447
    R[14] = (uint32_t)(hand >> 20);   // observation bits 448..479
}

// uniform random-legal action = k-th set bit of the mask, k = mulhi(r, n_legal).
// A legal mask is always {Pass, maybe X, maybe XX} + one contiguous run of bids up to
// 7NT, so the k-th set bit needs no bit-scan loop.
__device__ __forceinline__ int32_t kth_legal_action(uint64_t mask, uint32_t r) {
    uint32_t low = (uint32_t)mask & 7u;                 // Pass / X / XX
    uint32_t n_low = __popc(low);
    uint32_t bids = (uint32_t)(mask >> 3);              // 35 bid bits, bit b = bid b (low 32 here)
    uint32_t bids_hi = (uint32_t)(mask >> 35) & 7u;
    uint32_t first = bids ? (uint32_t)__ffs(bids) - 1u : (bids_hi ? 32u + (uint32_t)__ffs(bids_hi) - 1u : 35u);
    uint32_t n_legal = n_low + (35u - first);
    uint32_t k = __umulhi(r, n_legal);
    if (k >= n_low) return (int32_t)(3u + first + (k - n_low));
    // k-th set bit of a 3-bit field
    uint32_t b0 = low & 1u, b1 = (low >> 1) & 1u;
    if (k == 0u) return b0 ? 0 : (b1 ? 1 : 2);
    if (k == 1u) return (b0 && b1) ? 1 : 2;
    return 2;
}

__device__ __forceinline__ uint32_t action_uniform(uint64_t seed, uint64_t g, uint32_t step) {
    return philox4x32(make_uint4((uint32_t)g, (uint32_t)(g >> 32), kTagAct, step),
                      make_uint2((uint32_t)seed, (uint32_t)(seed >> 32))).x;
}

__device__ __forceinline__ int32_t random_legal_action(uint64_t mask, uint64_t seed, uint64_t g, uint32_t step) {
    return kth_legal_action(mask, action_uniform(seed, g, step));
}

}  // namespace brl
