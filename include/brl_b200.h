/*
 * brl_b200.h -- C ABI of the B200-native bridge-bidding environment path.
 *
 * The reference (harukaki/brl) has NO native/FFI layer: its boundary for this
 * path is the pgx 1.4.0 `bridge_bidding` Env Python surface used under
 * jax.jit / vmap / lax.scan (SURVEY 8b).  A jitted JAX program can only reach
 * CUDA through an XLA custom call, so every entry point below has exactly the
 * legacy XLA GPU custom-call shape
 *
 *     int32_t op(cudaStream_t stream, void **buffers,
 *                const void *opaque, size_t opaque_len);
 *
 * `buffers` = device pointers, inputs first then outputs, in the order listed
 * per op; `opaque` = one POD `BrlParams`.  The typed XLA FFI
 * (XLA_FFI_DEFINE_HANDLER) wraps the same symbols (csrc/xla_ffi_shim.cc,
 * INTEGRATION.md).  Rules for every op:
 *   - the caller owns every buffer; nothing is allocated, no stream is created,
 *     no host sync happens: the call only enqueues kernels on `stream` and is
 *     capturable in a CUDA graph / XLA command buffer;
 *   - optional outputs may be NULL (skipped); `state_in` may alias `state_out`
 *     (XLA input_output_aliases) -- every env is read before it is written;
 *   - re-entrant, no global mutable state;
 *   - returns 0 on success, a negative BRL_E_* on a usage error (bad opaque
 *     size, NULL required buffer, launch failure); `brl_last_error()` gives the
 *     message (thread-local).  Illegal ACTIONS are data, not errors: they
 *     terminate the env (SURVEY A.6.2).
 * There is no CPU fallback anywhere behind this ABI.
 *
 * Reference call sites each op replaces (paths relative to /root/reference):
 *   brl_init              env.init(key)                src/evaluation.py:95, ppo.py:305
 *   brl_step              env.step(state, action)      src/roll_out.py:51, src/duplicate.py:149
 *                         (+ BRL_F_AUTORESET: auto_reset wrapper src/utils.py:9-58)
 *   brl_duplicate_step    duplicate_step(env.step)     src/duplicate.py:147-192
 *   brl_duplicate_init    duplicate_init(state)        src/duplicate.py:132-135
 *   brl_observe           _observe(state, player)      src/duplicate.py:6,134
 *   brl_legal_mask        state.legal_action_mask      src/roll_out.py:78
 *   brl_rollout_random    act_randomly + auto_reset step, K steps per launch
 *                                                      src/duplicate.py:7,234 ; src/utils.py:9-58
 *   brl_imp_reward        _imp_reward                  src/duplicate.py:15-70
 *   brl_gae               calc_gae reverse scan        src/gae.py:20-39
 *   brl_categorical       masked distrax.Categorical   src/roll_out.py:27-30,79-81 ; src/evaluation.py:128-133
 *   brl_match_stats       mean / SE / win-rate sums    src/evaluation.py:199-201
 *   brl_state_fields      reads of State._dealer, ._last_bid, ... src/evaluation.py:97-112
 *   brl_reset_fields      State(...) construction / state.replace(...) src/duplicate.py:120-128
 *   brl_mlp_forward       forward.apply(params, obs) -> (logits, value)  src/models.py:23-33,
 *                         src/roll_out.py:73-76, src/utils.py:78-82, src/evaluation.py:124-127
 *   brl_policy_act        forward.apply + masked Categorical sample / mode + log_prob, fused   src/roll_out.py:73-81
 *   brl_ppo_loss          _loss_fn + jax.value_and_grad w.r.t. the net outputs   src/update.py:91-167
 *   brl_adam_clip         optimizer.update + optax.apply_updates                  src/update.py:168-169, ppo.py:195-211
 *   brl_adam_apply        the same with |grads|^2 taken from brl_ppo_grad (no pass over the gradient)
 *   brl_gather_rows       minibatch take(permutation)                             src/update.py:194-199
 *   brl_ppo_grad          jax.value_and_grad(_loss_fn)(params, traj, gae, targets) -> (loss_info, grads): minibatch
 *                         take + forward + loss + backward through the MLP on tcgen05   src/update.py:91-167,194-199
 *   brl_mlp_pack_train    flat fp32 params -> device layout for brl_ppo_grad
 *   brl_mlp_adam_step     optimizer.update + apply_updates + refresh of that layout, one pass   src/update.py:168-169
 *   brl_ppo_grad_grouped / brl_mlp_adam_step_grouped   the two above for K learners at once (population training)
 *   brl_ppo_grad_anchored / brl_ppo_grad_grouped_anchored   brl_ppo_grad(_grouped) + a KL penalty toward a fixed anchor policy
 *   brl_par / brl_gather_reward_par / brl_par_stats   not in the reference: the double-dummy par of each board, the
 *                         transition reward as IMPs against it, and a duplicate match's bidding against it (DESIGN.md f13)
 *   brl_system_stats / brl_system_stats_auctions   not in the reference: the hand strength and shape behind each call, by
 *                         net, context and call, counted in the match loop or over stored auctions (DESIGN.md f15)
 *   brl_call_values       not in the reference: every legal alternative of every decision of a duplicate match played out,
 *                         and the IMPs each would have changed, by net, context, played call and alternative (DESIGN.md f16);
 *                         optionally each decision's observation and gains as training examples (DESIGN.md f17)
 *   brl_cv_grad / brl_cv_eval   not in the reference: the all-actions policy-gradient loss head on those examples, on the
 *                         tensor-core forward / backward of brl_sl_grad (DESIGN.md f17)
 *   brl_hand_posterior    not in the reference: the hidden hands an auction implies under the nets' policies, by importance
 *                         sampling of the unseen cards with the grouped forward as the likelihood (DESIGN.md f18)
 *   brl_hand_posterior_smc  not in the reference: the same posterior by resample-move sequential Monte Carlo over the calls
 *                         of the auction (DESIGN.md f19)
 *   brl_eval_act_log      make_action + make_step_log of evaluate / duplicate_evaluate   src/evaluation.py:236-385, 650-745
 *   brl_eval_summary      make_terminated_log + the log_info means                        src/evaluation.py:448-596, 839-1027
 *   brl_mlp_pack          the params pytree (bridge_models/<name>.pkl, ppo.py:351-362) -> device layout
 *   brl_sl_examples       make_dataset: replay of a stored auction prefix -> (obs, legal mask, label)   sl.py:87-117
 *   brl_sl_grad           jax.value_and_grad(loss)(params, inputs, targets, legal_actions)             sl.py:169-184,205-206
 *   brl_sl_eval           loss + accuracy + illegal-action probability, no gradient                     sl.py:169-194,288-301
 *   brl_model_rows        the per-team net choice of every league match: live rows grouped by acting net
 *                                                      workspace/eval_selfplay_league.py ; src/evaluation.py:124-151
 *   brl_policy_act_grouped  team{1,2}_forward_pass.apply + masked argmax of every match of a league, one forward over a
 *                         pool of nets, row count read on the device   workspace/eval_selfplay_league.py ; src/evaluation.py:124-151
 *   brl_match_stats_ranges  brl_match_stats of every match of a league chunk   src/evaluation.py:199-201
 *   brl_duplicate_match   jax.jit(make_simple_duplicate_evaluate(...)) as one call: init, Table_info, the whole
 *                         lax.while_loop and the match sums   eval.py:53 ; src/evaluation.py:69-204
 *   brl_evaluate_match    jax.jit of make_evaluate's duplicate_evaluate / evaluate or of make_simple_evaluate as one call:
 *                         init, the whole lax.while_loop with the step log, and the log_info sums (or the actor's returns)
 *                         ppo.py:365-374 ; src/evaluation.py:11-66, 207-1032
 */
#ifndef BRL_B200_H
#define BRL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef BRL_CUDA_STREAM_T
#define BRL_CUDA_STREAM_T
typedef struct CUstream_st *brl_stream_t; /* == cudaStream_t */
#endif

#define BRL_ABI_VERSION 3
#define BRL_NUM_ACTIONS 38      /* 0 Pass, 1 X, 2 XX, 3..37 = 1C..7NT (src/duplicate.py:9-12) */
#define BRL_OBS_DIM 480         /* ppo.py:241, wb5/utils.py:48-52 */
#define BRL_NUM_PLAYERS 4
#define BRL_DEAL_ROW_BYTES 48   /* brl_b200/deals.py */
#define BRL_STATE_PLANES 5      /* packed state = uint4[BRL_STATE_PLANES][state_stride] */
#define BRL_STATE_BYTES_PER_ENV 80

/* flags */
#define BRL_F_AUTORESET     0x0001 /* src/utils.py:9-58 around the step */
#define BRL_F_RANDOM_ACTION 0x0002 /* draw a uniform random-legal action in-kernel (act_randomly) */
#define BRL_F_ACCUMULATE    0x0004 /* rewards += , terminated |= (quad step, src/utils.py:126-128) */
#define BRL_F_OBS_U8        0x0010 /* observation as bool/u8 (pgx dtype) instead of f32 */
#define BRL_F_OBS_BF16      0x0020 /* observation as bf16 (feeds a bf16 policy GEMM) */
#define BRL_F_SAMPLE        0x0040 /* brl_categorical: Gumbel-argmax sample instead of mode */
#define BRL_F_QUAD_LAST     0x0100 /* with ACCUMULATE: write the OR-ed terminated flag back into the state (src/utils.py:128) */
#define BRL_F_MLP_BF16      0x0200 /* brl_mlp_forward: one bf16 product per term instead of the 3-term split */
#define BRL_F_RESULT_I16    0x1000 /* brl_rollout_random: also write the compact result i16[K,n] into buffers[10] */
#define BRL_F_UNIFORM_U16   0x2000 /* brl_rollout_random / brl_env_rollout_host_compact*: caller-supplied uniforms are u16[K,n] */
#define BRL_F_SEED_SALT     0x4000 /* brl_policy_act: buffers[8] = device u64 XORed into `seed` (replayed CUDA graphs draw fresh noise) */
#define BRL_F_COUNT_DONE    0x8000 /* brl_gather_reward: buffers[3] u8 done[n], [4] inout u64 count += sum(done) (src/roll_out.py:85) */
#define BRL_F_SL_CHECK      0x0080 /* brl_sl_examples: replay every whole auction once and write a status byte per trajectory */
#define BRL_F_HOST_STAGED   0x0800 /* brl_env_create: never write results straight into pinned host buffers (always stage + copy) */

/* tuning (0 = automatic): bits 16-17 envs per block of the one-launch kernels (1->8, 2->16, 3->32), bits 18-19 warps
 * per block (1->1, 2->2, 3->4; 3 with bit 26: 8) */
#define BRL_F_TUNE_EPW(code) ((code) << 16)
#define BRL_F_TUNE_WPB(code) ((code) << 18)
#define BRL_F_TUNE_WPB8 ((3 << 18) | (1 << 26))
#define BRL_F_TUNE_CLASSIC_ROLLOUT (1 << 20)     /* tile-per-warp rollout kernel instead of the warp-specialised one */
#define BRL_F_TUNE_WRITERS(n) ((n) << 21)       /* writer warps (1..7) of the warp-specialised rollout; EPW bits = its envs per block */
/* the policy forward's path (brl_mlp_forward, brl_policy_act*), chosen by default by batch size: per-layer launches below
 * 4096 rows, one fused launch from 4096 on.  These bits share none with the env tuning bits above. */
#define BRL_F_TUNE_MLP_LAYERS (1 << 29)  /* per-layer launches at any size (BRL_F_SEED_SALT is then an error) */
#define BRL_F_TUNE_MLP_FUSED (1 << 30)   /* the fused launch at any size (ignored with BRL_F_TUNE_MLP_LAYERS) */

/* errors */
#define BRL_OK 0
#define BRL_E_OPAQUE (-1)   /* opaque_len != sizeof(BrlParams) or bad field */
#define BRL_E_BUFFER (-2)   /* required buffer is NULL / misaligned */
#define BRL_E_LAUNCH (-3)   /* CUDA launch error (message in brl_last_error) */
#define BRL_E_HANDLE (-4)   /* bad BrlEnv handle */

typedef struct BrlParams {
    int64_t n_envs;        /* envs in this call (this rank's shard); 0 = an empty batch: every batched op returns BRL_OK
                              without touching (or requiring) its buffers -- brl_team_rows still zeroes its counts */
    int64_t env_offset;    /* global index of env 0 (RNG counters use global indices)  */
    int64_t state_stride;  /* envs per plane of the packed state buffers (>= n_envs)   */
    uint64_t seed;         /* key of the counter-based action / Gumbel RNG             */
    int32_t n_deals;       /* rows in the deal table                                   */
    int32_t flags;         /* BRL_F_*                                                  */
    uint32_t step;         /* step counter of the action RNG (rollout: first step)     */
    int32_t k_steps;       /* rollout length K / GAE horizon T                         */
    float illegal_penalty; /* reward of a player making an illegal call (pgx: -1)      */
    float illegal_bonus;   /* reward of the three others                               */
    float gamma;           /* GAE                                                      */
    float gae_lambda;      /* GAE                                                      */
} BrlParams;

typedef int32_t (*brl_op_fn)(brl_stream_t, void **, const void *, size_t);

/* thread-local message of the last failing call on this thread ("" if none) */
const char *brl_last_error(void);
int32_t brl_abi_version(void);

/* buffers: [0] out u64 keys[n]
 * key_i = philox(seed, env_offset + i): mirrors jax.random.split(key, n). */
int32_t brl_make_keys(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* buffers: [0] in u64 keys[n]  [1] in deal_table
 *          [2] out state  [3] out obs[n,480]  [4] out u8 mask[n,38]  [5] out f32 rewards[n,4]
 *          [6] out u8 terminated[n]  [7] out i8 current_player[n] */
int32_t brl_init(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* Place envs on GIVEN episode draws.
 * buffers: [0] in i32 deal[n]  [1] in i32 dealer[n]  [2] in u8 vul_ns[n]  [3] in u8 vul_ew[n]
 *          [4] in i8 shuffled_players[n,4]  [5] in u64 rng_key[n] (NULL -> 0)  [6] in deal_table
 *          [7..12] out as brl_init [2..7] */
int32_t brl_reset_fields(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* buffers: [0] in state  [1] in i32 action[n] (ignored with BRL_F_RANDOM_ACTION)  [2] in deal_table
 *          [3] out state  [4] out obs  [5] out mask  [6] out rewards  [7] out terminated
 *          [8] out current_player  [9] out i32 action_taken[n] (optional) */
int32_t brl_step(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* Table_info = SoA {u8 terminated[n], f32 rewards[n,4], i32 last_bid[n], i32 last_bidder[n],
 *                   u8 call_x[n], u8 call_xx[n]}  (src/duplicate.py:138-144), updated in place.
 * buffers: [0] in state  [1] in action  [2] in deal_table
 *          [3..8] inout table A info  [9..14] inout table B info
 *          [15] out state  [16] out obs  [17] out mask  [18] out rewards  [19] out terminated
 *          [20] out current_player */
int32_t brl_duplicate_step(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* buffers: [0] in state  [1] in deal_table  [2..7] out as brl_init [2..7] */
int32_t brl_duplicate_init(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* buffers: [0] in state  [1] in i8 player_id[n] (NULL -> state.current_player)  [2] in deal_table
 *          [3] out obs */
int32_t brl_observe(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* buffers: [0] in state  [1] out u8 mask[n,38] */
int32_t brl_legal_mask(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* K auto-reset steps with in-kernel random-legal actions; every output is a
 * trajectory [K, n, ...] (any may be NULL); state updated in place.
 * buffers: [0] inout state  [1] in deal_table
 *          [2] out obs[K,n,480]  [3] out mask[K,n,38]  [4] out rewards[K,n,4]  [5] out terminated[K,n]
 *          [6] out current_player[K,n]  [7] out i32 action[K,n]
 *          [8] inout u64 stats[4] = {terminal steps, sum reward[player 0] (two's complement), calls, 0}
 *          [9] in u32 uniforms[K,n] (optional): caller-owned randomness; action = the
 *              mulhi(u, #legal)-th legal action.  NULL -> Philox(seed, env_offset+i, step+s).
 *              With BRL_F_UNIFORM_U16 the buffer is u16[K,n] and stands for the u32 uniform u16 << 16.
 *          [10] out i16 result[K,n] -- read ONLY with BRL_F_RESULT_I16: the step result in 2 bytes,
 *              result = 2 * rewards[player 0] + terminated.  Lossless on this path: pgx rewards are
 *              s * [+1,+1,-1,-1] by player id (players 0/1 partners) with s an integer duplicate score,
 *              |s| <= 7600, and random-legal play never takes the illegal-action branch.  Decode:
 *              terminated = result & 1, s = result >> 1 (arithmetic) -- brl_result16_decode. */
int32_t brl_rollout_random(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* buffers: [0] in f32 a_rewards[n,4]  [1] in f32 b_rewards[n,4]  [2] out f32 imp[n,4] */
int32_t brl_imp_reward(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* T = k_steps; all arrays time-major [T, n].
 * buffers: [0] in u8 done  [1] in f32 value  [2] in f32 reward  [3] in f32 last_val[n]
 *          [4] out f32 advantages  [5] out f32 targets */
int32_t brl_gae(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* buffers: [0] in f32 logits[n,38]  [1] in u8 mask[n,38] (NULL -> unmasked)
 *          [2] out i32 action[n]  [3] out f32 log_prob[n] */
int32_t brl_categorical(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* buffers: [0] in f32 x[n] (per-env return)  [1] inout f64 sums[8] += {n, sum x, sum x^2, #(x>0), 0,0,0,0} */
int32_t brl_match_stats(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* Unpack private fields (any output may be NULL).
 * buffers: [0] in state  [1] i32 deal  [2] i32 dealer  [3] i8 shuffled_players[n,4]  [4] u8 vul[n,2]
 *          [5] i32 last_bid  [6] i32 last_bidder  [7] u8 call_x  [8] u8 call_xx  [9] i32 pass_num
 *          [10] i32 step_count  [11] u64 rng_key */
int32_t brl_state_fields(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* Transition bookkeeping of roll_out._env_step (src/roll_out.py:85-94):
 * buffers: [0] in f32 rewards[n,4]  [1] in i8 actor[n]  [2] out f32 reward[n] = rewards[actor] / scale
 *          with BRL_F_COUNT_DONE: [3] in u8 done[n]  [4] inout u64 terminated_count[1] += sum(done)
 * scale passed in BrlParams.gamma. */
int32_t brl_gather_reward(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* Double-dummy par of each env's board (not in the reference; DESIGN.md f13 defines it): the minimax value of competitive
 * bidding over the deal row's DD table, with the env's dealer and vulnerability.
 * buffers: [0] in state (16-byte aligned)  [1] in deal_table
 *          [2] out f32 par[n,4] (16-byte aligned) in the rewards layout: by player id (p, p, -p, -p), p = par of the
 *              team of player ids {0, 1} under the state's seating
 *          [3] out i32 contract[n] (NULL ok): -1 passed out, else bid | declarer_seat << 8 | doubled << 10 */
int32_t brl_par(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* brl_gather_reward against par: reward = done ? IMP(rewards[actor] - par[actor]) / 24 : 0 (24 = the largest IMP).
 * buffers: [0] in f32 rewards[n,4]  [1] in i8 actor[n]  [2] in f32 par[n,4] (brl_par of the state before the step)
 *          [3] in u8 done[n]  [4] out f32 reward[n]
 *          [5] inout u64 terminated_count[1] += sum(done) -- read ONLY with BRL_F_COUNT_DONE (8-byte aligned)
 * rewards and par 16-byte aligned. */
int32_t brl_gather_reward_par(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* Bidding against par over the two tables of a duplicate match (brl_evaluate_match's Table_infos), for the team of player
 * ids {0, 1}: per table IMP(rewards[0] - par[0]), and whether the final contract is the par contract in level, strain and
 * declaring side (doubles ignored; two passed-out boards match).  Table B is table A's board with the teams' seats swapped.
 * buffers: [0] in state: table A's initial state (16-byte aligned)  [1] in deal_table
 *          [2] in f32 rewards_a[n,4]  [3] in i32 last_bid_a[n]  [4] in i32 last_bidder_a[n]
 *          [5] in f32 rewards_b[n,4]  [6] in i32 last_bid_b[n]  [7] in i32 last_bidder_b[n]
 *          [8] inout f64 sums[8] += {tables, sum imp, sum imp^2, sum |imp|, #par contract, 0, 0, 0}
 * rewards_a / rewards_b / sums 16-byte aligned.  The sums are integers: every order of addition gives the same result. */
int32_t brl_par_stats(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- policy / value net on the tensor cores (src/models.py:23-33, "DeepMind" 4x1024 ReLU) ----
 * Weights are packed once (transposed to K-major bf16 hi/lo pairs); the forward is five
 * TMA + tcgen05 GEMM launches with bias/ReLU/requantisation fused into the epilogues.
 * Default arithmetic: 3-term bf16 split accumulated in fp32 (fp32-class results);
 * BRL_F_MLP_BF16 = single bf16 product. */
int64_t brl_mlp_packed_bytes(void);
int64_t brl_mlp_scratch_bytes(int64_t n_envs);
/* buffers: [0..5] in f32 w_l[in,out] (haiku `linear`, `linear_1`..`linear_5`; y = x @ w + b)
 *          [6..11] in f32 b_l[out]   [12] out packed parameters (brl_mlp_packed_bytes()) */
int32_t brl_mlp_pack(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* buffers: [0] in obs[n,480] f32 (or u8 with BRL_F_OBS_U8)  [1] out bf16 obs[n,480] */
int32_t brl_obs_to_bf16(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* buffers: [0] in bf16 obs[n,480]  [1] in packed parameters  [2] scratch (brl_mlp_scratch_bytes(n))
 *          [3] out f32 logits[n,38]  [4] out f32 value[n] */
int32_t brl_mlp_forward(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* forward + masked categorical in one call -- `logits, value = forward.apply(params, obs); pi = Categorical(where(mask,
 * logits, -inf)); action = pi.sample(seed) | pi.mode(); log_prob = pi.log_prob(action)` (src/roll_out.py:73-81,
 * src/utils.py:78-88,150-160, src/evaluation.py:124-133).  From 4096 envs on this is ONE persistent launch: the thread
 * that drains a head-tile row holds its 38 logits and samples in place (same Philox noise as brl_categorical).
 * buffers: [0] in bf16 obs[n,480]  [1] in packed parameters  [2] scratch  [3] in u8 mask[n,38] (NULL -> unmasked)
 *          [4] out i32 action[n]  [5] out f32 log_prob[n] (NULL ok)  [6] out f32 value[n] (NULL ok)
 *          [7] out f32 logits[n,38] (NULL ok)  [8] in u64 seed_salt[1] -- read ONLY with BRL_F_SEED_SALT
 * params: flags BRL_F_SAMPLE / BRL_F_MLP_BF16, seed, env_offset, step as for brl_categorical. */
int32_t brl_policy_act(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* brl_policy_act on a LIST of envs: n_envs = number of listed rows.  obs / mask / action / log_prob are the full per-env
 * arrays; only the listed envs are read and written.  This is how the evaluation loops (src/evaluation.py:124-151) avoid
 * the reference's vmap waste of running both teams' nets on every env and of forwarding finished envs.
 * buffers: [0] in bf16 obs[total,480]  [1] in packed parameters  [2] scratch (brl_mlp_rows_scratch_bytes(n_envs))
 *          [3] in u8 mask[total,38] (NULL -> unmasked)  [4] out i32 action[total]  [5] in i32 row_index[n_envs]
 *          [6] out f32 log_prob[total] (NULL ok)  [7] out f32 logits[total,38] (NULL ok; rows of the listed envs)
 * The Gumbel noise of BRL_F_SAMPLE is keyed by env_offset + row_index[r], i.e. identical to the unlisted call. */
int64_t brl_mlp_rows_scratch_bytes(int64_t n_rows);
int32_t brl_policy_act_rows(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* Rows of the envs still playing, split by the team of the player to act (players 0/1 = team 1, 2/3 = team 2).
 * buffers: [0] in i8 current_player[n]  [1] in u8 done[n] (NULL -> all live)  [2] out i32 rows_team1[n]
 *          [3] out i32 rows_team2[n]  [4] out i32 counts[2] */
int32_t brl_team_rows(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- self-play league over a pool of M nets (workspace/eval_selfplay_league.py; each match src/evaluation.py:69-204) ----
 * All matches of the league run as one batch of envs.  The pool is M packed blobs (brl_mlp_pack) stacked
 * brl_mlp_pool_stride() bytes apart.  Every live env is forwarded by the net that acts there: brl_model_rows groups the rows
 * by net and writes the padded row count offsets[M] to device memory, and brl_policy_act_grouped runs all nets in one forward
 * that reads that count on the device, so a step needs no host read.  brl_duplicate_match plays a whole match this way.
 * BrlParams.k_steps = M in both. */
int64_t brl_mlp_pool_stride(void);
/* rows a grouping of n_envs envs over M nets can need: each non-empty group is padded to 256 rows (one row tile) */
int64_t brl_model_rows_capacity(int64_t n_envs, int64_t n_models);
/* k_team_rows generalised (src/evaluation.py:124-151 with a net per env and team): env i is live unless done[i]; its acting
 * net is env_models[i][0] for players 0/1 and env_models[i][1] for players 2/3.  A live env whose id is outside [0, M) is an
 * error: offsets[M] comes back as -1 (the host reads offsets[M] anyway to size the forward; the other outputs are then invalid).
 * buffers: [0] in i8 current_player[n]  [1] in u8 done[n] (NULL -> all live)  [2] in i32 env_models[n,2]
 *          [3] out i32 rows[brl_model_rows_capacity(n, M)]: net m's live envs at [offsets[m], offsets[m] + counts[m]), then -1
 *              up to offsets[m + 1]  [4] out i32 counts[M]  [5] out i32 offsets[M + 1] (multiples of 256; offsets[M] = the
 *              padded row count)  [6] out i32 block_model[capacity / 256]: the net of each 256-row block
 * An empty batch (n_envs = 0) zeroes counts / offsets when they are given.
 * BRL_F_PLAYER_MODELS: [2] is i32 env_models[n,4] by player id instead, and env i's acting net is env_models[i][player]
 * (the two partners of a team may be different nets); the bad-id rule is the same. */
#define BRL_F_PLAYER_MODELS (1 << 24)  /* brl_model_rows / brl_duplicate_match: a net per player id, env_models[n,4] */
int32_t brl_model_rows(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* brl_policy_act_rows with the net of each row block taken from the pool (masked argmax only; BRL_F_SAMPLE is an error).
 * The row count n_rows[0] (offsets[M] of brl_model_rows, e.g. a pointer to offsets + M) is read on the device only: the call
 * is sized for n_envs rows, and the rows from n_rows[0] on are not read.  Action and logits of the listed envs are written by env.
 * buffers: [0] in bf16 obs[total,480]  [1] in pool u8[M, brl_mlp_pool_stride()]  [2] scratch (brl_mlp_rows_scratch_bytes(n_envs),
 *          = brl_policy_grouped_scratch_bytes(total, M) for the capacity)  [3] in u8 mask[total,38] (NULL -> unmasked)
 *          [4] out i32 action[total]  [5] in i32 rows[n_envs]  [6] in i32 block_model[n_envs / 256]
 *          [7] out f32 logits[total,38] (NULL ok)  [8] in i32 n_rows[1] (4-byte aligned)
 * params: n_envs = the capacity of rows (a multiple of 256, e.g. brl_model_rows_capacity(total, M)), k_steps = M, flags
 *         BRL_F_MLP_BF16 / BRL_F_TUNE_MLP_LAYERS / BRL_F_TUNE_MLP_FUSED.  The path is brl_policy_act's rule on n_envs (one fused
 *         launch from 4096 on, per-layer launches below), so n_envs = n_rows[0] runs the path of that batch size.
 * rows / block_model / n_rows must be brl_model_rows' output for the same M, with n_rows[0] <= n_envs: they are device data and
 * not checked here; a block id outside [0, M) or a count above n_envs is undefined behaviour. */
int64_t brl_policy_grouped_scratch_bytes(int64_t n_envs, int64_t n_models);
int32_t brl_policy_act_grouped(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* brl_match_stats over P = n_envs contiguous ranges (the matches of a league chunk), each entry exactly what brl_match_stats
 * gives on that slice.  buffers: [0] in f32 x  [1] in i64 offsets[P + 1] (range p = [offsets[p], offsets[p + 1]))
 *          [2] inout f64 sums[P, 8] */
int32_t brl_match_stats_ranges(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- a whole duplicate match as one call (eval.py:53, src/evaluation.py:69-204) ---------------------------------------
 * make_simple_duplicate_evaluate's duplicate_evaluate for every env of the batch, with the loop on the device:
 *   brl_init from the keys (:93-95) -> Table_info A = B from the init state (:97-112) -> while any env is live { live rows
 *   grouped by acting net (brl_model_rows, :124-151) -> masked-argmax forward of every net of the pool
 *   (brl_policy_act_grouped, :124-133) -> brl_duplicate_step (:164) -> cum_return += rewards[:, 0] (:167-169) } ->
 *   sums += brl_match_stats per env range (:199-201).
 * The loop is a CUDA graph WHILE node whose condition a kernel sets from the padded row count on the device; the forward
 * takes its row count from device memory too, and its path follows brl_policy_act's rule on that count (one fused launch
 * from 4096 rows on, per-layer launches below; BRL_F_TUNE_MLP_LAYERS / BRL_F_TUNE_MLP_FUSED pin one).  Nothing is read
 * back to the host.  On a plain stream the call captures the match once per set of buffers and params into a graph it
 * keeps (repeated calls with the same buffers relaunch it; brl_duplicate_match_graph_builds() counts the builds); on a
 * stream that is being captured (a CUDA graph, an XLA command buffer) it adds the same nodes to the caller's capture.
 * Unlike the other ops it keeps this cache and three private capture streams per device, created on the first call;
 * make that first call outside a capture.
 * buffers: [0] in u64 keys[n] (brl_make_keys)  [1] in deal_table  [2] in pool u8[M, brl_mlp_pool_stride()]
 *          [3] in i32 env_models[n,2] (NULL: M must be 2, every env plays net 0 on players 0/1 against net 1 on 2/3)
 *          [4] in i64 range offsets[P + 1] (NULL: one range, the whole batch)  [5] scratch
 *          (brl_duplicate_match_scratch_bytes(n, M))  [6] out f32 cum_return[n]  [7] inout f64 sums[P, 8] (+=, as
 *          brl_match_stats_ranges; sums[8] for one range)  [8] out i32 status[1] (BRL_MATCH_*)
 *          [9..14] out final Table_info A {u8 terminated, f32 rewards[n,4], i32 last_bid, i32 last_bidder, u8 call_x,
 *          u8 call_xx}  [15..20] out Table_info B -- all twelve or none (then they live in the scratch)
 *          [21] inout u32 system_hist[M, 75, 38, 96] (NULL: not counted): each iteration runs brl_system_stats between the
 *          grouped forward and brl_duplicate_step, on the forward's actions and this call's env_models (by team or by player),
 *          so every decision of the match is counted for the net that made it.  Without it the graph is the one without
 *          the histogram.  The XLA form keeps the 21-buffer layout: [21] is NULL there.
 * params: n_envs = n, k_steps = M, step = P (0 with [4] NULL), n_deals, illegal_penalty / illegal_bonus as brl_step,
 *         flags BRL_F_MLP_BF16 / BRL_F_TUNE_MLP_LAYERS / BRL_F_TUNE_MLP_FUSED (BRL_F_SAMPLE is an error).
 * BRL_F_PLAYER_MODELS: [3] is a required i32 env_models[n,4] by player id (brl_model_rows' flag; NULL is BRL_E_BUFFER), so
 * each player of a match may be a different net: partnerships of two nets (cross-play).  Player ids keep their team at both
 * tables (table B swaps seats, not ids), so the ids need no change at the table switch. */
#define BRL_MATCH_MAX_STEPS 638    /* an auction has at most 319 calls; an env finishes both tables in at most 638 steps */
#define BRL_MATCH_OK 0
#define BRL_MATCH_BAD_MODEL 1      /* a live env's acting net id is outside [0, M): the loop stopped, outputs invalid */
#define BRL_MATCH_STEP_BOUND 2     /* envs still live after BRL_MATCH_MAX_STEPS forwards: the loop stopped */
int64_t brl_duplicate_match_scratch_bytes(int64_t n_envs, int64_t n_models);
long long brl_duplicate_match_graph_builds(void);
int32_t brl_duplicate_match(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- a whole evaluation as one call (ppo.py:365-374; src/evaluation.py:11-66, 207-1032) ----------------------------------
 * brl_duplicate_match's device loop (WHILE node, control kernel, path kernel and IF nodes, graph cache, adding to a caller's
 * capture, BRL_MATCH_* status and bound) for the other evaluators of ppo.train.  The pool holds two nets: net 0 is team 1 /
 * the actor, net 1 team 2 / the opponent.  The mode is flags bits 27-28 (BRL_F_EVAL_MATCH(m)):
 *   BRL_EVAL_MATCH_DUPLICATE  make_evaluate(duplicate=True)'s duplicate_evaluate (:615-1027): brl_init (:617-619) ->
 *       Table_info A = B (:621-636) -> while any env is live { brl_model_rows -> grouped forward with the logits by env ->
 *       brl_eval_act_log (:650-745) -> brl_duplicate_step (:772-774) -> cum_return += rewards[:, 0] (:775-777) } ->
 *       brl_state_fields (step_count) -> brl_eval_summary with both Table_infos into sums (:839-1027).
 *   BRL_EVAL_MATCH_SINGLE  make_evaluate(duplicate=False)'s evaluate (:256-596): the same loop with brl_step (no auto-reset,
 *       :406) and rewards_sum += rewards, cum_return += rewards[:, 0] (:407-411); brl_eval_summary takes the final state's
 *       fields (:448-596); BRL_F_EVAL_INDICATOR_BIDS is implied (:345-354).
 *   BRL_EVAL_MATCH_SIMPLE  make_simple_evaluate (:11-66): every decision is an argmax and the net acting is fixed per seat, so
 *       the quad step (src/utils.py:133-202) is one env step per iteration: net 0 decides for the team of the env's INITIAL
 *       current_player, net 1 for the other team; R[i] += rewards[i, initial player] per step (rewards are non-zero only on
 *       the terminal step, so this is the per-quad sum).  The output is R[n] in [4]; the caller takes R.mean().
 * BRL_F_EVAL_FREE_RUN (full statistics only, game_mode "free-run"): team 2 always passes.  Every live row is forwarded by net 0
 * (team 2's too: brl_model_rows needs no change) and brl_eval_act_log reads no team-2 logits, so the results equal the host
 * loop's at the cost of forwarding team 2's rows; net 1 is not read.
 * BRL_F_EVAL_PARTNER: the pool holds 3 nets (k_steps = 3): net 0 is the actor, net 1 team 2 and net 2 the actor's partner,
 * grouped by player id (BRL_F_PLAYER_MODELS).  DUPLICATE / SINGLE: player 0 plays net 0, player 1 net 2, players 2/3 net 1.
 * SIMPLE: the env's initial current_player plays net 0, that player's partner net 2 and the other team net 1.  With
 * BRL_F_EVAL_FREE_RUN team 2 still passes and net 1 is not read: team 2's rows are forwarded by net 0, team 1's are split
 * between nets 0 and 2.  The scratch is brl_evaluate_match_partner_scratch_bytes(n, mode).
 * buffers: [0] in u64 keys[n]  [1] in deal_table  [2] in pool u8[2, brl_mlp_pool_stride()]
 *          [3] scratch (brl_evaluate_match_scratch_bytes(n, mode))  [4] out f32 cum_return[n] (simple: R[n])
 *          [5] out f32 acc[n, BRL_EVAL_ACC_COLS] (full statistics; simple: not read)
 *          [6] inout f64 sums[239] (+= brl_eval_summary; simple: not read)  [7] out i32 status[1] (BRL_MATCH_*)
 *          [8..13] out final Table_info A, [14..19] B, as brl_duplicate_match [9..20] (duplicate mode: all twelve or none)
 *          [20] out final state  [21] out bf16 obs[n,480]  [22] out u8 mask[n,38]  [23] out f32 rewards_sum[n,4]
 *          [24] out u8 terminated[n]  [25] out i8 current_player[n] (single-table mode: all six or none; the state after the
 *          loop with rewards = the summed rewards, what evaluate returns, :591)
 * Buffers a mode does not read may be NULL.  Without [8..19] / [20..25] those live in the scratch.
 * params: n_envs = n, n_deals, illegal_penalty / illegal_bonus as brl_step, flags BRL_F_EVAL_MATCH(mode) |
 *         BRL_F_EVAL_FREE_RUN | BRL_F_MLP_BF16 | BRL_F_TUNE_MLP_LAYERS / BRL_F_TUNE_MLP_FUSED (BRL_F_SAMPLE is an error).
 * The graph cache and brl_duplicate_match_graph_builds() are shared with brl_duplicate_match. */
#define BRL_EVAL_MATCH_DUPLICATE 1
#define BRL_EVAL_MATCH_SINGLE 2
#define BRL_EVAL_MATCH_SIMPLE 3
#define BRL_F_EVAL_MATCH(mode) ((mode) << 27)
#define BRL_EVAL_MATCH_MODE(flags) (((flags) >> 27) & 3)
#define BRL_F_EVAL_FREE_RUN 0x0008
#define BRL_F_EVAL_PARTNER (1 << 25)  /* brl_evaluate_match: a 3-net pool, net 2 the actor's partner */
int64_t brl_evaluate_match_scratch_bytes(int64_t n_envs, int64_t mode);
int64_t brl_evaluate_match_partner_scratch_bytes(int64_t n_envs, int64_t mode);
int32_t brl_evaluate_match(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- bidding-system statistics (not in the reference; DESIGN.md f15, restated by tests/system_ref.py) --------------------
 * A decision is one call a (BRL_NUM_ACTIONS numbering) of the player at seat s.  Its context c in [0, 75) depends only on the
 * earlier calls of the auction (call k made by seat (dealer + k) mod 4):
 *   c = t        OPEN(t), t = 0..3: every earlier call is Pass (t = the caller's position after the dealer)
 *   c = 4 + b    RESPONSE(b): the only bid so far is bid b (0..34), made by the caller's partner two calls ago; the call since
 *                was Pass; no X / XX
 *   c = 39 + b   OVERCALL(b): the only bid so far is bid b, made by the caller's right-hand opponent at the previous call
 *   c = 74       OTHER
 * Hand features of seat s from the deal row: HCP (A 4, K 3, Q 2, J 1; 0..37), suit lengths (clubs, diamonds, hearts,
 * spades), balanced = no void or singleton and at most one doubleton (4333, 4432, 5332).
 * hist[M, 75, 38, 96] u32 (+=), per net m, context c and call a: columns 0..37 the HCP histogram, 38 + 14 * suit + length the
 * suit-length histograms, 94 the balanced hands, 95 the decisions (1,094,400 bytes per net).  A call adds one to at most seven
 * cells per decision it counts, so a cell stays exact while hist plus the call's decisions stays below 2^32; callers that
 * accumulate longer add each call's histogram into a wider one. */
#define BRL_SYS_CONTEXTS 75
#define BRL_SYS_COLS 96
/* One decision per live env, in the state before the step: the call action[i] of the player to act, into the histogram of the
 * net acting there by brl_model_rows' rule (env_models by team, or by player with BRL_F_PLAYER_MODELS; NULL: net 0 for every
 * env).  Calls outside 0..37 and net ids outside [0, M) are not counted.  One thread per env, global atomics into the
 * (L2-resident) histogram.
 * buffers: [0] in state (16-byte aligned)  [1] in deal_table  [2] in i32 action[n]  [3] in u8 done[n] (NULL: all live)
 *          [4] in i32 env_models[n, 2] by team or [n, 4] by player id with BRL_F_PLAYER_MODELS (NULL: net 0)
 *          [5] inout u32 hist[M, 75, 38, 96]
 * params: n_envs, state_stride (0: n_envs), k_steps = M, flags BRL_F_PLAYER_MODELS. */
int32_t brl_system_stats(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* Every call of stored auctions, the context read from the call sequence (no env replay): auction t is calls[offsets[t],
 * offsets[t + 1]) (brl_sl_examples' encoding) on deal row board[t] with dealer dealer[t].  Calls must be in 0..37 and rows in
 * the table: they are not checked here.
 * buffers: [0] in deal_table  [1] in u8 calls[]  [2] in i64 offsets[n + 1]  [3] in i32 board[n] (NULL: row t)
 *          [4] in i8 dealer[n] (NULL: North, the convention of the OpenSpiel data files)  [5] inout u32 hist[1, 75, 38, 96]
 * params: n_envs = n auctions. */
int32_t brl_system_stats_auctions(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- counterfactual call values (not in the reference; DESIGN.md f16, restated by tests/call_values_ref.py) --------------
 * The base match is the duplicate match brl_duplicate_match plays for the same keys, pool, env_models and flags; every
 * decision is the masked argmax of the acting net.  A decision d is each step where env e is live at table T (A or B): the
 * pre-step state S_d, the player p to act and its net m (brl_model_rows' rule), the context c of brl_system_stats, and the
 * played call b_d.  For every call a legal in S_d the branch (d, a) starts from brl_step(S_d, a) (no auto-reset, no table
 * switch) and plays that one table to its end, each player acting with its own net from env_models (masked argmax); r_d(a)
 * is the branch's final rewards[0].  With R_A, R_B the base match's final rewards[0] at both tables:
 *   gain   g_d(a) = sigma_p * (imp_of_difference(r_d(a) + R_other) - imp_of_difference(R_A + R_B)), sigma_p = +1 for players
 *          0/1, -1 for 2/3: the change of the decider's team's match IMPs with the other table held at its result, in [-48, 48]
 *   regret regret_d = max over legal a of g_d(a) >= 0 (a hindsight bound: the decider does not see the other hands)
 * The played branch is the base game, so r_d(b_d) = R_T; the op counts the decisions where it is not (`mismatch`).
 * Per base iteration the body forwards the base envs, writes 38 branch slots per env (an illegal call's or a finished env's
 * slot is born finished), plays them out in a nested WHILE node (grouping by player, grouped forward, brl_step, control with a
 * bound of 319 calls per auction), forms the gains, and only then steps the base envs with brl_duplicate_step.
 * buffers: [0] in u64 keys[n]  [1] in deal_table  [2] in pool u8[M, brl_mlp_pool_stride()]
 *          [3] in i32 env_models[n, 2] by team (or [n, 4] by player id with BRL_F_PLAYER_MODELS), 16-byte aligned
 *          [4] in f32 rewards_a[n, 4], [5] in f32 rewards_b[n, 4]: the final Table_info rewards of brl_duplicate_match on the
 *          same keys, nets and flags  [6] scratch (brl_call_values_scratch_bytes(n, M))
 *          [7] out i64 gain_sums[M, 75, 38, 38, 4] = {n, sum g, sum g^2, #(g > 0)} per (net, context, played, alternative)
 *          [8] out i64 regret_sums[M, 75, 4] = {decisions, sum regret, sum regret^2, #(regret > 0)}
 *          [9] out i64 mismatch[M]: decisions with r_d(b_d) != R_T  [10] out i32 status[1] (BRL_MATCH_*)
 *          [11] out i64 count[1] (the decisions, also beyond the capacity)  [12..17] out i32 env (env_offset + i), table (0 A,
 *          1 B), player, net, context, played [cap]  [18] out f32 r[cap, 38] (NaN for an illegal call) -- the records, all
 *          eight or none
 *          [19] out bf16 obs[cap, 480]: the observation row the acting net's forward read at record k's decision
 *          [20] out f32 gain[cap, 38]: record k's g_d(a), NaN exactly where the call is illegal -- the training examples of
 *          DESIGN.md f17 (row k belongs to record k), both or neither, and only with the records; obs 16-byte aligned.
 *          Without them the graph is the one without the feature; through the XLA target they are NULL.
 * params: n_envs = n, k_steps = M, n_deals, env_offset (added to the records' env), seed = the record capacity cap,
 *         illegal_penalty / illegal_bonus, flags BRL_F_PLAYER_MODELS | BRL_F_MLP_BF16 | BRL_F_TUNE_MLP_* (BRL_F_SAMPLE is an
 *         error).  More decisions than cap set BRL_MATCH_RECORD_CAPACITY; the sums stay complete.  An empty batch is a
 *         no-op.  The graph cache and capture rules are brl_duplicate_match's. */
#define BRL_MATCH_RECORD_CAPACITY 3  /* brl_call_values: more decisions than record slots; every sum is still complete */
int64_t brl_call_values_scratch_bytes(int64_t n_envs, int64_t n_models);
int32_t brl_call_values(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- hand reading (not in the reference; DESIGN.md f18, restated by tests/posterior_ref.py) -----------------------------
 * What an observer can infer about the three hidden hands from an auction, under the nets' own policies.
 * Auctions use brl_system_stats_auctions' encoding: auction t is calls[offsets[t], offsets[t + 1]) (calls 0..37) on deal row
 * board[t] (NULL: row t) with dealer dealer[t] (NULL: North) and vulnerability vul[t] (bit 0 NS, bit 1 EW; NULL: none); call k
 * is made by seat (dealer + k) mod 4.  Query j = query[j] = (t, s, L): auction t, the observer's absolute seat s, the prefix
 * length L (0 <= L <= the auction's length).  seat_nets[j, 0..3] = the net of each absolute seat, an index into a pool of M
 * packed nets brl_mlp_pool_stride() bytes apart.
 *   Sample i of query j (global index g = env_offset + j): the 39 cards outside the observer's hand, in increasing card index
 *   h[0..38], are shuffled by Fisher-Yates: for t = 0..37, with n = 38 - t, swap h[n] and h[mulhi(u_t, n + 1)], where u_t is
 *   word (t mod 4) (x, y, z, w) of philox4x32(counter (g_lo, g_hi, BRL_POST_TAG + t / 4, i), key (seed_lo, seed_hi)).  Then
 *   h[0..12] are the observer's left-hand opponent's (seat s + 1), h[13..25] partner's (s + 2), h[26..38] the right-hand
 *   opponent's (s + 3).  The samples depend on (seed, g, i) only.
 *   Likelihood: for every k < L whose caller sigma_k != s, o is sigma_k's observation after c_0 .. c_{k-1} (vulnerability and
 *   history relative to sigma_k, sigma_k's hand from the sample), m its legal mask, l the logits of net seat_nets[j, sigma_k]
 *   on o (bf16 observation, the grouped forward).  l_k = log softmax over the legal calls of l / tau at c_k, in f32 as
 *   brl_categorical forms log_prob (x - max - log sum exp); with tau = 0, l_k = 0 when c_k is the masked argmax (first maximum)
 *   and -inf otherwise.  log w[j, i] = sum of l_k in f64, k increasing.
 *   Posterior (self-normalised importance weights under the uniform prior): M_j = max_i log w, w' = exp(log w - M_j),
 *   W = sum w'.  cards[j, r, c] = sum w' [card c held by relative seat r] / W (r = 0 LHO, 1 partner, 2 RHO);
 *   features[j, r, 0..94] = the w'-weighted distribution of that hand's features in brl_system_stats' columns (HCP 0..37,
 *   38 + 14 suit + length, 94 balanced) / W; weights[j] = {M_j, W, sum w'^2, #(w > 0)} (ESS = W^2 / sum w'^2).  Every sum is f64
 *   over i increasing, so the outputs are bit-identical across runs, chunkings and batch compositions.  A query without an
 *   accepted sample, or with a status other than BRL_POST_OK, has NaN cards / features / weights[0..2] and a count of 0.
 * The call: a check pass (one thread per (query, k)), the row layout (segment (j, k) = N consecutive rows, one per sample, in
 * its net's group; groups padded to 256 rows, the padded count in device memory), the public pass (each segment's rotated
 * history words, vulnerability bits, legal mask and call), the sampler, the observation expansion (bf16 rows, only the hand
 * bits vary in a segment), the grouped forward of brl_policy_act_grouped with logits out (its path by brl_policy_act's rule on
 * the row capacity: pass the exact padded row count to run the path of that count), the per-sample log-likelihood and a
 * per-query reduction.  No host synchronisation; capturable.
 * buffers: [0] in deal_table  [1] in u8 calls[]  [2] in i64 offsets[]  [3] in i32 board[] (NULL: row t)  [4] in i8 dealer[]
 *          (NULL: North)  [5] in u8 vul[] (NULL: none)  [6] in i32 query[Q, 3]  [7] in i32 seat_nets[Q, 4]
 *          [8] in pool u8[M, brl_mlp_pool_stride()]  [9] scratch (brl_hand_posterior_scratch_bytes(Q, N, capacity, M))
 *          [10] out f64 cards[Q, 3, 52]  [11] out f64 features[Q, 3, 95]  [12] out f64 weights[Q, 4]  [13] out i32 status[Q]
 *          [14] out u64 hands[Q, N, 4] by absolute seat  [15] out f64 logw[Q, N] -- diagnostics, both or neither
 * params: n_envs = Q, env_offset = the global index of query 0, seed, step = N (samples per query, 1 .. 2^24), k_steps = M,
 *         state_stride = the row capacity (a multiple of 256), n_deals = rows in the deal table, gamma = tau (>= 0; < 0 or NaN
 *         is BRL_E_OPAQUE), flags BRL_F_MLP_BF16 | BRL_F_TUNE_MLP_LAYERS / BRL_F_TUNE_MLP_FUSED.  t must name an auction of the
 *         buffers and calls must be in 0..37: they are not checked here.  An empty batch is a no-op. */
#define BRL_POST_TAG 0x484E4430u  /* "HND0": Philox stream of the hand sampler, + block index 0..9 */
#define BRL_POST_OK 0
#define BRL_POST_ILLEGAL 1        /* a call of the prefix is not legal where it is made */
#define BRL_POST_SHORT 2          /* the auction ends before call L, or L is longer than the auction */
#define BRL_POST_BAD_NET 3        /* a seat that calls in the prefix (not the observer) has a net id outside [0, M) */
#define BRL_POST_BAD_QUERY 4      /* s outside 0..3, L < 0, or the deal row outside the table */
#define BRL_POST_CAPACITY 5       /* the layout needs more rows than the capacity: every query of the call, outputs invalid */
#define BRL_POST_FEATURES 95
int64_t brl_hand_posterior_scratch_bytes(int64_t n_queries, int64_t n_samples, int64_t row_capacity, int64_t n_models);
int32_t brl_hand_posterior(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- hand reading by resample-move SMC (not in the reference; DESIGN.md f19, restated by tests/smc_ref.py) ---------------
 * The query of brl_hand_posterior, answered by sequential Monte Carlo over the calls of the prefix (Gilks & Berzuini 2001;
 * Del Moral, Doucet & Jasra 2006), so that long and informative auctions keep an effective sample size.
 *   Particles i = 0..N-1 of query g start as brl_hand_posterior's samples; each carries its hidden hands, log w (f64, 0) and
 *   ell[r] (f64, 0), the sum of its l_k over the calls of hidden seat r (0 LHO, 1 partner, 2 RHO).  Stage k = 0 .. K-1
 *   (K = `stages` >= every query's L): a stage with k >= L, a call by the observer, or an extinct query does nothing.  Else,
 *   sigma_k the caller:
 *   1. reweight: l_k is brl_hand_posterior's term of call k on the particle's hands; log w += l_k, ell[sigma_k] += l_k.
 *   2. resample: M = max log w; if M = -inf the query is extinct for good.  w' = exp(log w - M), W = sum w', S = sum w'^2 (i
 *      increasing).  When kappa = 1 or W * W / S < kappa * N: systematic resampling with u = (x + 0.5) 2^-32, x = word x of
 *      philox4x32(counter (g_lo, g_hi, BRL_SMC_TAG + 128 k, 0xFFFFFFFF), key (seed_lo, seed_hi)): C_m = C_{m-1} + w'_m (i
 *      increasing, C_0 = w'_0); the ancestor of particle i is the first m with C_m >= (i + u) * W / N (at most N - 1).  Hands
 *      and ell are copied from the ancestors, log_evidence += log(W / N) + M, log w = 0, resamples += 1.
 *   3. move, after a resample only, for mv = 0 .. R-1: with P = philox4x32(counter (g_lo, g_hi, BRL_SMC_TAG + 128 k + 1 + mv,
 *      c3), key): the pair is mulhi(P(c3 = 0xFFFFFFFF).x, 3) (0: LHO + partner, 1: LHO + RHO, 2: partner + RHO), shared by the
 *      query; particle i (c3 = i) swaps card mulhi(P.x, 13) of r1 with card mulhi(P.y, 13) of r2 (the n-th card in increasing
 *      card index).  ell'[r] = the sum of the proposed hands' l over seat r's calls at stages <= k (k increasing); accepted iff
 *      log((P.z + 0.5) 2^-32) < (ell'[r1] + ell'[r2]) - (ell[r1] + ell[r2]), then hands and ell[r1], ell[r2] take the proposal.
 *   4. end: brl_hand_posterior's reduction of log w; log_evidence += log(W / N) + M (-inf when nothing is accepted).
 *   Every draw depends on (seed, g, k, mv, i) only, so results do not depend on batching.  With kappa = 0 no query resamples
 *   and cards, features, weights, status, hands and log w are those of brl_hand_posterior bit for bit, on a pinned forward path.
 * The call enqueues per stage: the row layout of call k of every live query, f18's public pass, expansion and grouped forward,
 * the reweight, the ESS test / resampling (one thread per query), the gather; per move the proposal, the layout of the pair's
 * calls at stages <= k for the queries that resampled, the forward and the MH test.  Row counts stay in device memory; no host
 * synchronisation; capturable.  The row capacity bounds each forward, not their sum.
 * buffers: [0]-[13] as brl_hand_posterior; [9] scratch (brl_hand_posterior_smc_scratch_bytes(Q, N, capacity, M))
 *          [14] out f64 log_evidence[Q] (NaN on a status other than OK)  [15] out i32 resamples[Q]
 *          [16] out f64 acceptance[Q] (accepted / proposed moves; NaN with none proposed)
 *          [17] out u64 hands[Q, N, 4]  [18] out f64 logw[Q, N]  [19] out f64 ell[Q, N, 3] -- final particles, all or none
 *          [20] out f64 trace_loglik[Q, K, N] (l_k, NaN when stage k does nothing)  [21] out i32 trace_ancestors[Q, K, N]
 *          (-1 without a resample)  [22] out i32 trace_pairs[Q, K, R] (-1 without a move)  [23] out u8 trace_accepted[Q, K, R, N]
 *          [24] out f64 trace_proposed[Q, K, R, N, 2] (ell'[r1], ell'[r2]) -- the trace, all five or none
 * params: BrlSmcParams: post as brl_hand_posterior's BrlParams; ess_threshold = kappa in [0, 1]; moves = R in [0, 64];
 *         stages = K in [0, 320]; reserved = 0.  A query with L > K gets BRL_POST_STAGES. */
#define BRL_SMC_TAG 0x534D0000u  /* "SM": Philox stream of the SMC draws, + 128 k + (0 | 1 + mv) */
#define BRL_POST_STAGES 6         /* brl_hand_posterior_smc: the prefix is longer than the stage bound */
#define BRL_SMC_MAX_MOVES 64
#define BRL_SMC_MAX_STAGES 320
typedef struct BrlSmcParams {
    BrlParams post;       /* brl_hand_posterior's parameters */
    float ess_threshold;  /* kappa: resample when ESS < kappa N; 1 resamples at every stage */
    int32_t moves;        /* R: Metropolis-Hastings moves after each resample */
    int32_t stages;       /* K: the stage bound */
    int32_t reserved;     /* 0 */
} BrlSmcParams;
int64_t brl_hand_posterior_smc_scratch_bytes(int64_t n_queries, int64_t n_samples, int64_t row_capacity, int64_t n_models);
int32_t brl_hand_posterior_smc(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- PPO update, non-GEMM part (src/update.py:74-242, ppo.py:195-211) ----------------------- */
#define BRL_PPO_VALUE_CLIPPING  0x1 /* config["value_clipping"]  (src/update.py:47-62) */
#define BRL_PPO_REWARD_SCALING  0x2 /* config["reward_scaling"]: (gae - mean) / (std + 1e-8) per minibatch (src/update.py:31-45) */
#define BRL_PPO_UNMASKED_POLICY 0x4 /* actor_illegal_action_penalty mode: log-prob from the unmasked softmax (src/update.py:18-24) */
#define BRL_PPO_ILLEGAL_STAT    0x8 /* brl_ppo_grad with illegal_l2_coef == 0: also form the logged illegal_action_loss (a 38 x 38
                                       eigen-problem per minibatch, ~19 us); clear: stats[6] = NaN.  With a non-zero coefficient
                                       and in brl_ppo_loss the norm is always formed (the gradient needs it). */

typedef struct BrlPpoParams {
    int64_t batch;         /* samples in this minibatch                                  */
    int64_t total;         /* rows of the flat [T * n_envs] trajectory the index addresses */
    float clip_eps;        /* config["clip_eps"]                                         */
    float ent_coef;        /* config["ent_coef"]                                         */
    float vf_coef;         /* config["vf_coef"]                                          */
    float illegal_l2_coef; /* config["illegal_action_l2norm_coef"]                       */
    int32_t flags;         /* BRL_PPO_*                                                  */
    int32_t reserved;      /* 0.  brl_ppo_grad reads experiment bits here (0 = measured defaults): 4 / 16 = the other tile
                              width (128x128 / 128x64) in the fused forward / backward launch, 8 = per-tile time stamps
                              into the scratch (brl_mlp_train_trace_offset) */
} BrlPpoParams;

#define BRL_PPO_SCRATCH_BYTES 188416 /* scratch of brl_ppo_loss / brl_ppo_grad (buffers[12]) */

typedef struct BrlAdamParams {
    int64_t n;             /* elements of the flat parameter buffer                      */
    int32_t step;          /* 1-based optimizer step count (bias correction)             */
    float lr;              /* learning rate for THIS step (schedules are evaluated by the caller, ppo.py:186-192) */
    float beta1, beta2, eps; /* optax.adam defaults 0.9 / 0.999, eps = 1e-5 (ppo.py:198) */
    float max_grad_norm;   /* optax.clip_by_global_norm; <= 0 disables                   */
} BrlAdamParams;

/* _loss_fn of src/update.py:91-162 from the logits / value the net produced for one minibatch, fused
 * with its backward: d total_loss / d logits and d total_loss / d value come out of the same pass.
 * opaque = BrlPpoParams.
 * buffers: [0] in f32 logits[B,38]  [1] in f32 value[B]  [2] in i32 index[B] (row of each sample in the
 *          flat trajectory; NULL = identity)  [3] in u8 mask[total,38]  [4] in i32 action[total]
 *          [5] in f32 old_log_prob[total]  [6] in f32 old_value[total]  [7] in f32 advantages[total]
 *          [8] in f32 targets[total]  [9] out f32 dlogits[B,38]  [10] out f32 dvalue[B]
 *          [11] out f32 stats[8] = {total_loss, value_loss, loss_actor, entropy, approx_kl, clipfracs,
 *               illegal_action_loss, 0 (the anchor KL of brl_ppo_grad_anchored)}  [12] scratch, BRL_PPO_SCRATCH_BYTES, 16-byte aligned (f64[16] accumulators, then the
 *               38 x 38 Gram partials of the illegal-probability matrix: illegal_action_loss is its SPECTRAL norm / 2,
 *               jnp.linalg.norm(X, ord=2) of a 2-D array, src/update.py:141-142) */
int32_t brl_ppo_loss(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* optax.chain(clip_by_global_norm(max_grad_norm), adam(lr, eps)) over one flat fp32 buffer.  opaque = BrlAdamParams.
 * buffers: [0] inout f32 params[n]  [1] in f32 grads[n]  [2] inout f32 m[n]  [3] inout f32 v[n]  [4] scratch f64[1] */
int32_t brl_adam_clip(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* brl_adam_clip with the gradient's sum of squares supplied by the caller: [4] in f64[1] sum g^2 (brl_ppo_grad leaves it in
 * element 14 of its f64[16] scratch, accumulated by the weight- and bias-gradient epilogues), no extra pass over the gradient. */
int32_t brl_adam_apply(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* minibatch gather (jnp.take(x, permutation, axis=0), src/update.py:194-199): n_envs = B rows, k_steps = bytes per row.
 * buffers: [0] in src[total, row]  [1] in i32 index[B]  [2] out dst[B, row] */
int32_t brl_gather_rows(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- PPO update, the trip through the net (src/update.py:91-167): forward + backward on tcgen05 ---- */
#define BRL_PPO_OBS_U8   0x10 /* brl_ppo_grad: trajectory observations are u8 / bool 0-1 (pgx dtype) */
#define BRL_PPO_OBS_BF16 0x20 /* brl_ppo_grad: trajectory observations are bf16 (what the tensor-core rollout records) */
/* Flat fp32 parameter / gradient buffer: haiku modules actor_critic/linear, linear_1 .. linear_5 in that order, each
 * w[in,out] then b[out] (480x1024, 3 x 1024x1024, 1024x38, 1024x1): brl_mlp_num_params() = 3,681,319 floats. */
int64_t brl_mlp_num_params(void);
int64_t brl_mlp_train_blob_bytes(void);
int64_t brl_mlp_train_scratch_bytes(int64_t batch);
int64_t brl_mlp_train_trace_offset(int64_t batch); /* debug: offset in the scratch of the u64[2][4096][8] tile time stamps written when
                                                        BrlPpoParams.reserved bit 3 is set (scripts/exp_train_trace.py) */
/* flat params -> training blob: per layer (4 hidden + the 64-wide policy/value head tile) W[in, out_pad] as bf16 hi / lo in
 * haiku's own orientation -- the forward reads it as an MN-major tensor-core operand, the input-gradient GEMM as a K-major
 * one, so training keeps ONE copy of the weights and never transposes -- and the bias in fp32.  Needed once per parameter
 * set; inside the update loop brl_mlp_adam_step keeps the blob current.  opaque = BrlParams (fields unused).
 * buffers: [0] in f32 params[brl_mlp_num_params()]  [1] out blob[brl_mlp_train_blob_bytes()] */
int32_t brl_mlp_pack_train(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* optimizer.update + optax.apply_updates (src/update.py:168-169, ppo.py:195-211) for the flat MLP parameters, with the
 * refreshed parameters written into the training blob in the same pass: brl_adam_apply + brl_mlp_pack_train as one kernel.
 * opaque = BrlAdamParams (n = brl_mlp_num_params()).
 * buffers: [0] inout f32 params[n]  [1] in f32 grads[n]  [2] inout f32 m[n]  [3] inout f32 v[n]
 *          [4] in f64[1] sum of squares of grads (element 14 of brl_ppo_grad's scratch)  [5] inout blob */
int32_t brl_mlp_adam_step(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* One minibatch of `jax.value_and_grad(_loss_fn, has_aux=True)(params, traj_batch, gae, targets)` (src/update.py:164-167):
 * take(index) of the observations, forward with the activations kept, brl_ppo_loss, backward GEMMs (input gradients with
 * the ReLU mask fused, weight gradients contracted over the batch, bias gradients), all products as three-term bf16
 * splits accumulated in fp32 on the tensor cores.  opaque = BrlPpoParams (flags: BRL_PPO_* incl. BRL_PPO_OBS_*).
 * buffers: [0] in obs[total,480] (f32 unless BRL_PPO_OBS_*)  [1] in blob (brl_mlp_pack_train)
 *          [2] scratch[brl_mlp_train_scratch_bytes(B)]  [3] in i32 index[B] (NULL = identity)  [4] in u8 mask[total,38]
 *          [5] in i32 action[total]  [6] in f32 old_log_prob[total]  [7] in f32 old_value[total]
 *          [8] in f32 advantages[total]  [9] in f32 targets[total]  [10] out f32 grads[brl_mlp_num_params()]
 *          [11] out f32 stats[8] (as brl_ppo_loss)  [12] scratch, BRL_PPO_SCRATCH_BYTES (as brl_ppo_loss); on return its f64
 *               element 14 = sum of squares of grads (the input of brl_adam_apply) */
int32_t brl_ppo_grad(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* brl_ppo_grad with a KL penalty toward a fixed anchor policy: the loss gains kl_coef * mean_b KL(pi(.|s_b) || alpha(.|s_b)),
 * pi the policy distribution of the loss (masked softmax, or the unmasked one with BRL_PPO_UNMASKED_POLICY), alpha the
 * softmax of the anchor's logits over the same action set (0 log 0 := 0).  d / d logit_j = kl_coef / B * pi_j (log pi_j -
 * log alpha_j - KL_b) on the set, 0 elsewhere.  opaque = BrlPpoParams.
 * buffers: [0..12] as brl_ppo_grad  [13] in f32 anchor_logits[total, 38] (the anchor net's logits for each trajectory row)
 *          [14] in f32 kl_coef[1] (device scalar)
 * stats[0] includes kl_coef * KL, stats[7] = mean_b KL_b.  With kl_coef = 0 the gradient and stats[0..6] are bit-equal to
 * brl_ppo_grad's.  An empty batch (batch = 0) is a no-op and its buffers may be NULL. */
int32_t brl_ppo_grad_anchored(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- population training: one optimizer step of K learners in the launches of one ------------------------------------
 * K PPO learners of the same shape (minibatch size B, flags) each take their step on their own weights, trajectory and
 * coefficients.  The GEMM tiles of all learners share one fused forward and one fused backward launch, so that one
 * learner's dependency gaps are filled by the others' tiles.  Learner k's gradient, stats and |g|^2 are bit-identical to
 * a brl_ppo_grad call with its inputs (same tile widths, K-block order and epilogue arithmetic); its |g|^2 is a sum of
 * f64 atomics and may differ in the last bits.  An empty batch (n_learners = 0 or batch = 0) is a no-op and its buffers
 * may be NULL. */
#define BRL_MAX_LEARNERS 64
/* floats between two learners' rows of a population's flat parameter / gradient / moment buffers [K, stride]: the row
 * is brl_mlp_num_params() floats padded to 256 bytes (the padding is neither read nor written) */
int64_t brl_mlp_param_stride(void);
typedef struct BrlPpoGroupedParams {
    int64_t batch;         /* samples in each learner's minibatch (one B for all)                                        */
    int32_t n_learners;    /* K, 0 .. BRL_MAX_LEARNERS                                                                   */
    int32_t flags;         /* BRL_PPO_* incl. BRL_PPO_OBS_*, the same for all learners                                    */
    int32_t reserved;      /* 0; bits 2 / 4 pick the fused launches' tile widths as in BrlPpoParams.reserved (bit 3 unused) */
    int32_t pad;           /* 0 */
} BrlPpoGroupedParams;
int64_t brl_ppo_grad_grouped_scratch_bytes(int64_t n_learners, int64_t batch);
/* brl_ppo_grad for K learners.  opaque = BrlPpoGroupedParams.  Learner k's rows of a [K, ...] buffer are its own.
 * buffers: [0] in i64 traj[K, 8]: device addresses of learner k's obs[total_k, 480] (dtype per BRL_PPO_OBS_*), i32 index[B]
 *              (NULL = identity), u8 mask[total_k, 38], i32 action, f32 old_log_prob, old_value, advantages, targets [total_k]
 *              -- the buffers of brl_ppo_grad, one allocation per learner; 16-byte aligned table
 *          [1] in f32 coefs[K, 4] = {clip_eps, ent_coef, vf_coef, illegal_l2_coef} per learner
 *          [2] in blob[K, brl_mlp_train_blob_bytes()]  [3] scratch[brl_ppo_grad_grouped_scratch_bytes(K, B)]
 *          [4] out f32 grads[K, brl_mlp_param_stride()]  [5] out f32 stats[K, 8] (as brl_ppo_grad)
 *          [6] scratch acc[K, BRL_PPO_SCRATCH_BYTES]; on return learner k's f64 element 14 = its |grads|^2
 * Buffers [2], [3], [4] and [6] are 16-byte aligned.  Undefined: a table address that is not a valid buffer of the size
 * above, an index outside [0, total_k), buffers that overlap. */
int32_t brl_ppo_grad_grouped(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* brl_ppo_grad_anchored for K learners.  opaque = BrlPpoGroupedParams.
 * buffers: [0..6] as brl_ppo_grad_grouped  [7] in i64 anchor_logits[K]: device address of learner k's f32 anchor logits
 *          [total_k, 38]  [8] in f32 kl_coef[K]
 * Learner k's results are bit-identical to a brl_ppo_grad_anchored call with its inputs.  An empty batch is a no-op. */
int32_t brl_ppo_grad_grouped_anchored(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* brl_mlp_adam_step for K learners in one launch.  opaque = BrlAdamParams[K] (opaque_len = K * sizeof, 0 = no-op): learner
 * k's step count, learning rate, betas, eps and max_grad_norm; n = brl_mlp_num_params() for every k.
 * buffers: [0] inout f32 params[K, s]  [1] in f32 grads[K, s]  [2] inout f32 m[K, s]  [3] inout f32 v[K, s], s =
 *              brl_mlp_param_stride()  [4] in acc[K, BRL_PPO_SCRATCH_BYTES] of brl_ppo_grad_grouped (learner k's |grads|^2: its f64 element 14)
 *          [5] inout blob[K, brl_mlp_train_blob_bytes()]; all 16-byte aligned */
int32_t brl_mlp_adam_step_grouped(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- supervised bidding pre-training (sl.py): examples from stored auctions, cross-entropy step ---------------------- */
/* Examples of the OpenSpiel bidding data (sl.py:87-117): one deal row per trajectory (deals.py format, DD nibbles unused),
 * dealer North, nobody vulnerable, players = seats (bridge(use_double_dummy_result=false), sl.py:44).  The calls of
 * trajectory t are calls[offsets[t] .. offsets[t + 1]) as actions 0..37 (0 Pass, 1 X, 2 XX, 3.. = 1C..7NT).
 * opaque = BrlParams: n_envs = examples B (check mode: trajectories to check), n_deals = trajectories in the table,
 *          flags = BRL_F_OBS_U8 / BRL_F_OBS_BF16 (f32 default) | BRL_F_SL_CHECK, seed / step / env_offset key the positions.
 * buffers: [0] in deal_table[n_deals, 48]  [1] in u8 calls[]  [2] in i64 offsets[n_deals + 1]  [3] in i32 traj[B]
 *          [4] in i32 position[B] (call index in [0, n_calls); NULL -> uniform from Philox(seed; env_offset + b, step))
 *          [5] out obs[B,480] of the player to act after calls [0, position)  [6] out u8 mask[B,38]
 *          [7] out i32 label[B] = the call at `position` (-1: position outside the auction)  [8] out i32 position[B] (NULL ok)
 *          [9] out u8 status[n_envs] -- written ONLY with BRL_F_SL_CHECK (then [3..8] are not read or written):
 *              BRL_SL_* for trajectory i's whole auction */
#define BRL_SL_OK        0 /* legal throughout, ends with its last call */
#define BRL_SL_ILLEGAL   1 /* a call that is not legal where it is made */
#define BRL_SL_EARLY_END 2 /* the auction is over before its last call */
#define BRL_SL_NOT_ENDED 3 /* the auction is not over after its last call */
int32_t brl_sl_examples(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

typedef struct BrlSlParams {
    int64_t batch;         /* examples in this minibatch; 0 = an empty batch (no-op)      */
    float ent_coef;        /* SLConfig.entropy_coef                                      */
    int32_t flags;         /* BRL_F_OBS_U8 / BRL_F_OBS_BF16: dtype of obs (f32 default)   */
} BrlSlParams;
#define BRL_SL_ACC_BYTES 128 /* f64[16] accumulators of brl_sl_grad / brl_sl_eval; element 14 = sum of squares of grads */

/* One minibatch of `jax.value_and_grad(loss, has_aux=True)` (sl.py:169-184, 205-206) through the DeepMind MLP on tcgen05
 * (the forward / backward of brl_ppo_grad with a cross-entropy head):
 *   target_loss = -mean(one_hot(label, 38) * log_softmax(logits)) (mean over B * 38 entries, unmasked softmax),
 *   entropy of the softmax over the legal calls, total = target_loss - ent_coef * entropy; the value head gets no gradient.
 * Follow with brl_mlp_adam_step, eps = 1e-8, max_grad_norm = 0 (optax.adam(learning_rate), sl.py:166).  opaque = BrlSlParams.
 * buffers: [0] in obs[B,480]  [1] in blob (brl_mlp_pack_train)  [2] scratch[brl_mlp_train_scratch_bytes(B)]
 *          [3] in u8 mask[B,38]  [4] in i32 label[B]  [5] out f32 grads[brl_mlp_num_params()]
 *          [6] out f32 stats[8] = {total_loss, target_loss, entropy, accuracy, illegal_actions_prob, 0, 0, 0}
 *          [7] scratch f64[16] (BRL_SL_ACC_BYTES, 16-byte aligned) */
int32_t brl_sl_grad(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* brl_sl_grad's forward and statistics without the backward (the post-update train accuracy, sl.py:279, and the test
 * metrics, sl.py:288-301): accuracy = mean(argmax softmax(logits) == label), illegal_actions_prob = mean(softmax . ~legal).
 * buffers: [0] in obs  [1] in blob  [2] scratch  [3] in u8 mask[B,38]  [4] in i32 label[B]  [5] out f32 stats[8]  [6] scratch f64[16] */
int32_t brl_sl_eval(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- call-value policy improvement (not in the reference; DESIGN.md f17, restated by tests/cvi_ref.py) -----------------
 * An all-actions policy-gradient step on brl_call_values' training examples: sample b has the gains g[b, a] of every call
 * (NaN: illegal; the legal set is isfinite(g)).  pi = softmax of the logits over the legal calls, gbar = sum_a pi_a g_a,
 * J_b = gbar / 24 (the IMP scale of reward_mode "par_imp"), H_b = entropy of pi.
 *   loss = -mean_b J_b - ent_coef * mean_b H_b
 *   d loss / d l_j = -pi_j (g_j - gbar) / (24 B) + ent_coef * pi_j (log pi_j + H_b) / B for legal j, 0 otherwise; the value
 *   head gets no gradient.  A sample without a legal call contributes 0 to everything and 1 to stat 6.
 * Follow with brl_mlp_adam_step.  opaque = BrlSlParams (batch, ent_coef, flags BRL_F_OBS_U8 / BRL_F_OBS_BF16, and the
 * experiment bits BRL_CV_WIDE_FORWARD / BRL_CV_NARROW_BACKWARD: the other tile width of the fused forward (128x128) /
 * backward (128x64) launch, as BrlPpoParams.reserved bits 4 / 16; 0 = the measured defaults).
 * buffers: [0] in obs[B,480]  [1] in blob (brl_mlp_pack_train)  [2] scratch[brl_mlp_train_scratch_bytes(B)]
 *          [3] in f32 gain[B,38]  [4] out f32 grads[brl_mlp_num_params()]
 *          [5] out f32 stats[8] = {total loss, mean gbar (IMPs), mean g of the argmax-logit legal call (lowest index on
 *              ties), mean (max_a g_a - that gain), mean entropy, share of samples whose argmax-logit call has the maximal g,
 *              mean unmasked-softmax mass on illegal calls, 0}
 *          [6] scratch f64[16] (BRL_SL_ACC_BYTES, 16-byte aligned; element 14 = sum of squares of grads) */
#define BRL_CV_WIDE_FORWARD    (1 << 16)
#define BRL_CV_NARROW_BACKWARD (1 << 17)
int32_t brl_cv_grad(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* brl_cv_grad's forward and statistics without the backward (the same stats, bit for bit).
 * buffers: [0] in obs  [1] in blob  [2] scratch  [3] in f32 gain[B,38]  [4] out f32 stats[8]  [5] scratch f64[16] */
int32_t brl_cv_eval(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* ---- full evaluation statistics (src/evaluation.py:207-1032) ---------------------------------- */
#define BRL_F_EVAL_INDICATOR_BIDS 0x0400 /* non-duplicate `evaluate`: bid histogram is .set(1), not += 1 (src/evaluation.py:345-354) */
#define BRL_EVAL_ACC_COLS 76    /* per-env log row: ill[2] steps[2] passes[2] actor_bid[35] opp_bid[35] (team 1 first) */
int32_t brl_eval_num_sums(void); /* length of the partial-sum vector of brl_eval_summary (239) */
/* One evaluation step: action = masked argmax of the ACTING team's logits (team 1 = players 0/1) and the
 * per-env log update of update_log_info, skipped for finished envs.
 * buffers: [0] in f32 logits_team1[n,38]  [1] in f32 logits_team2[n,38] (NULL = free-run opponent: always Pass)
 *          [2] in u8 mask[n,38]  [3] in i8 current_player[n]  [4] in u8 terminated[n]
 *          [5] out i32 action[n]  [6] inout f32 acc[n,76] */
int32_t brl_eval_act_log(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);
/* End of match: every mean of the log_info tuple as f64 partial sums (sums += ...; all-reduce, then divide).
 * sums layout: [0] n [1] sum cum [2] sum cum^2 [3] #(cum>0) [4] sum ill1/steps1 [5] sum ill2/steps2 [6] sum step_count
 *   [7] sum pass1/steps1 [8] sum pass2/steps2 [9] sum tableA rewards[0] [10] sum tableB rewards[0]
 *   [11+9t ..] per table t: pass_out, x1, xx1, x2, xx2, make1, make2, down1, down2
 *   [29..98] bid histograms team 1 then team 2   [99+70t ..] contract histograms of table t, team 1 then team 2
 * buffers: [0] in f32 acc[n,76]  [1] in f32 cum_return[n]  [2] in i32 step_count[n]
 *          [3..8] table A: i32 last_bid, i32 last_bidder, u8 call_x, u8 call_xx, f32 rewards[n,4] (NULL: sign from
 *                 cum_return), i32 pass_num (NULL: not required for a pass-out)
 *          [9..14] table B likewise ([9] NULL = single-table evaluate)   [15] inout f64 sums[239] */
int32_t brl_eval_summary(brl_stream_t, void **buffers, const void *opaque, size_t opaque_len);

/* -------------------------------------------------------------------------
 * Legacy XLA GPU custom-call targets (API_VERSION_STATUS_RETURNING -- the convention
 * of jax/jaxlib 0.4.23, the version brl pins in requirements.txt:25-26).  `buffers` arrive in
 * XLA's order -- the op's inputs (operands) first, then its outputs (results), each in the
 * order the op documents; a buffer the op updates in place is an operand AND an aliased result
 * (input_output_aliases) -- and are re-ordered into the op's list by csrc/xla_ffi_shim.cc from
 * the per-op layout string `brl_xla_layout(name)` returns (one char per op buffer: i input,
 * o output, s scratch output, x in place).  `opaque` = the bytes of the op's params struct.  A
 * failing op sets the XLA status through XlaCustomCallStatusSetFailure, looked up in the process
 * at call time; without that symbol the failure is counted in brl_xla_unreported_failures() and
 * stays in brl_last_error().  Register with xla_client.register_custom_call_target(name,
 * capsule, "CUDA") (INTEGRATION.md).  Typed-FFI handlers `<op>_ffi` for the same table are built
 * only when the XLA FFI headers are present.
 * ------------------------------------------------------------------------- */
const char *brl_xla_layout(const char *op_name);
long long brl_xla_unreported_failures(void);
struct XlaCustomCallStatus_;
void brl_make_keys_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_init_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_reset_fields_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_step_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_duplicate_step_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_duplicate_init_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_observe_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_legal_mask_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_rollout_random_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_imp_reward_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_gae_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_categorical_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_match_stats_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_state_fields_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_gather_reward_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_mlp_pack_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_obs_to_bf16_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_mlp_forward_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_policy_act_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_policy_act_rows_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_team_rows_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_model_rows_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_policy_act_grouped_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_match_stats_ranges_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_duplicate_match_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_evaluate_match_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_ppo_loss_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_adam_clip_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_adam_apply_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_gather_rows_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_mlp_pack_train_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_mlp_adam_step_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_ppo_grad_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_ppo_grad_grouped_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_ppo_grad_anchored_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_ppo_grad_grouped_anchored_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_mlp_adam_step_grouped_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_eval_act_log_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_eval_summary_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_sl_examples_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_sl_grad_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_sl_eval_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_par_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_gather_reward_par_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_system_stats_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_system_stats_auctions_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_call_values_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_cv_grad_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_cv_eval_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_par_stats_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_hand_posterior_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);
void brl_hand_posterior_smc_xla(brl_stream_t, void **buffers, const char *opaque, size_t opaque_len, struct XlaCustomCallStatus_ *status);

/* -------------------------------------------------------------------------
 * Host-buffer convenience layer (the call a non-JAX host makes): the library
 * owns device state + pinned staging; inputs/outputs are HOST pointers and the
 * copies are part of the call.  Synchronous.  Used for bench.py's `e2e`.
 * ------------------------------------------------------------------------- */
typedef struct BrlEnv BrlEnv;

BrlEnv *brl_env_create(int64_t n_envs, int64_t env_offset, const uint8_t *deal_table_host,
                       int32_t n_deals, uint64_t seed, int32_t flags);
void brl_env_destroy(BrlEnv *env);
/* init from philox keys of (seed, env_offset+i); outputs as brl_env_step_host */
int32_t brl_env_init_host(BrlEnv *env, void *obs, uint8_t *mask, float *rewards, uint8_t *terminated,
                          int8_t *current_player);
/* action: host i32[n] (NULL with BRL_F_RANDOM_ACTION); outputs: host buffers (any may be NULL).
 * obs dtype follows the env's flags (f32 default, BRL_F_OBS_U8 = pgx bool). */
int32_t brl_env_step_host(BrlEnv *env, const int32_t *action, void *obs, uint8_t *mask, float *rewards,
                          uint8_t *terminated, int8_t *current_player);
/* One rollout of k_steps auto-reset random-legal steps (the shape of roll_out's scan,
 * src/roll_out.py:105).  HOST in: uniforms u32[k_steps, n] (the randomness of the action
 * choice; NULL -> in-kernel Philox).  HOST out (any may be NULL): rewards f32[k_steps,n,4],
 * terminated u8[k_steps,n], stats u64[4] (as brl_rollout_random).  The observation / mask
 * trajectories stay in HBM for a device-resident consumer, exactly as `traj_batch` does in
 * the reference; `brl_env_trajectory` exposes their device pointers.
 * If `rewards` / `terminated` are pinned host memory the kernel writes them in place over PCIe
 * (no copy phase); pageable buffers are staged in HBM and copied under the next chunk of steps. */
int32_t brl_env_rollout_host(BrlEnv *env, int32_t k_steps, const uint32_t *uniforms, float *rewards,
                             uint8_t *terminated, uint64_t *stats);
/* Pipelined form: enqueue and return a ticket (> 0; negative = BRL_E_*).  Call c's input copy runs under call
 * c-1's kernel and its result copy under call c+1's kernel.  The host buffers of a call are valid after
 * brl_env_wait(env, ticket); keep at most BRL_ENV_PIPELINE_DEPTH calls in flight, each with its own set of host
 * buffers.  Three in flight keep the GPU fed (with two, the host learns that D2H(c-1) finished only as kernel c
 * ends -- too late to enqueue c+1 without a bubble). */
#define BRL_ENV_PIPELINE_DEPTH 4
int64_t brl_env_rollout_host_async(BrlEnv *env, int32_t k_steps, const uint32_t *uniforms, float *rewards,
                                   uint8_t *terminated, uint64_t *stats);
int32_t brl_env_wait(BrlEnv *env, int64_t ticket);
/* Compact-payload forms (same rollout, same device-resident trajectory incl. f32 rewards / u8 terminated, see
 * brl_env_trajectory): what crosses PCIe is 2 bytes per env-step each way instead of 4 in + 17 out.
 * HOST in: uniforms u32[k_steps,n], or u16[k_steps,n] when the env was created with BRL_F_UNIFORM_U16 (NULL -> in-kernel
 * Philox).  HOST out: result i16[k_steps,n] = 2 * rewards[player 0] + terminated (lossless, see brl_rollout_random
 * buffers[10]; this is what roll_out's consumer reads: rewards[actor] and done, src/roll_out.py:86-94), stats u64[4].
 * Tickets share brl_env_wait and the BRL_ENV_PIPELINE_DEPTH staging slots with brl_env_rollout_host_async. */
int64_t brl_env_rollout_host_compact_async(BrlEnv *env, int32_t k_steps, const void *uniforms, int16_t *result,
                                           uint64_t *stats);
int32_t brl_env_rollout_host_compact(BrlEnv *env, int32_t k_steps, const void *uniforms, int16_t *result, uint64_t *stats);
/* host-side decode of `rows` compact results into rewards f32[rows,4] / terminated u8[rows] (either may be NULL) */
void brl_result16_decode(const int16_t *result, int64_t rows, float *rewards, uint8_t *terminated);
/* device pointers of the last rollout's trajectory: obs, mask, rewards, terminated, current_player, action */
int32_t brl_env_trajectory(BrlEnv *env, void **out_ptrs6);

/* -------------------------------------------------------------------------
 * Trajectory memory.  Observation and mask rows are almost all zero bytes; on
 * memory mapped with generic compression the L2 compresses such lines on their
 * way to DRAM, which shrinks a rollout's write-back.  brl_alloc_compressible
 * reserves address space, creates a physical allocation (compressible when
 * CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED says the device has it,
 * a plain one otherwise), maps it read/write for `device` and returns its
 * address; NULL on failure (brl_last_error).  The size is rounded up to the
 * allocation granularity.  *granted (may be NULL) = 1 when the driver granted
 * compression.  brl_free_compressible synchronises the device (as cudaFree
 * does) and unmaps; NULL and unknown pointers are ignored.  The host-buffer
 * layer's obs / mask trajectories come from here.
 * ------------------------------------------------------------------------- */
void *brl_alloc_compressible(size_t bytes, int32_t device, int32_t *granted);
void brl_free_compressible(void *ptr);
/* granularity brl_alloc_compressible rounds to on `device` (bytes; -1 on error) */
int64_t brl_compressible_granularity(int32_t device);
/* bytes rounded up to a multiple of granularity (granularity 0: bytes) */
size_t brl_round_up_granularity(size_t bytes, size_t granularity);

#ifdef __cplusplus
}
#endif
#endif /* BRL_B200_H */
