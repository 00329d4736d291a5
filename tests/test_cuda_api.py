"""GPU parity of the host-side mirror of the reference interface (BridgeBidding / State,
auto_reset + quad steps, make_roll_out, make_calc_gae, duplicate evaluation) against the
oracle, on the SAME deals, DD tables and ACTION SEQUENCES (north star): the loops run on
the GPU, every action they took is replayed through the oracle, and everything the env
produced must match bit-exactly.  Action choice itself (an fp32 GEMM + masked argmax /
Gumbel sample) is checked separately against a NumPy MLP with a near-tie report."""
import numpy as np
import pytest
import torch

from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _mk_env(n_deals=3000, seed=2, **kw):
    from brl_b200 import BridgeBidding
    from brl_b200.deals import synthetic_deal_table
    table = synthetic_deal_table(n_deals, seed=seed)
    return BridgeBidding(table=table, device=DEV, **kw), table


def test_env_surface_shapes_dtypes_and_private_fields():
    from oracle import oracle as orc
    env, table = _mk_env()
    n = 300
    assert env.observation_shape == (480,) and env.num_actions == 38
    keys = env.make_keys(5, n)
    state = env.init(keys)
    assert state.observation.shape == (n, 480) and state.observation.dtype == torch.float32
    assert state.legal_action_mask.dtype == torch.bool and state.legal_action_mask.shape == (n, 38)
    assert state.rewards.shape == (n, 4) and state.terminated.dtype == torch.bool
    assert state.current_player.dtype == torch.int8 and not state.truncated.any()
    ref = orc.OracleEnv(table, n)
    ref.init(keys.cpu().numpy().view(np.uint64))
    p = ref.export_private()
    assert (state._dealer.cpu().numpy() == p["dealer"]).all()
    assert (state._shuffled_players.cpu().numpy() == p["shuffled_players"]).all()
    assert (state._vul_NS.cpu().numpy() == p["vul"][:, 0].astype(bool)).all()
    assert (state._last_bid.cpu().numpy() == -1).all() and (state._last_bidder.cpu().numpy() == -1).all()
    assert (state._pass_num.cpu().numpy() == 0).all() and (state._step_count.cpu().numpy() == 0).all()
    # functional step: the input state is untouched
    before = state._packed.clone()
    nxt = env.step(state, torch.zeros(n, dtype=torch.int32, device=DEV))
    assert (state._packed == before).all() and (nxt._step_count.cpu().numpy() == 1).all()
    ref.step(np.zeros(n, np.int32))
    assert (nxt.observation.cpu().numpy() == ref.export()["observation"]).all()


def test_act_randomly_is_uniform_over_legal_actions():
    from brl_b200 import act_randomly
    env, _ = _mk_env()
    n = 20000
    state = env.init(env.make_keys(1, n))
    state = env.step(state, torch.full((n,), 10, dtype=torch.int32, device=DEV))  # everyone's dealer bids 2H
    a = act_randomly(123, state).cpu().numpy()
    mask = state.legal_action_mask.cpu().numpy()
    assert mask[np.arange(n), a].all()
    legal = np.flatnonzero(mask[0])
    freq = np.bincount(a, minlength=38)[legal] / n
    assert np.abs(freq - 1.0 / len(legal)).max() < 0.01


def _replay_quads(ref, trace, n):
    """Replay traced sub-step actions (4 per quad) through the oracle's auto-reset step;
    returns per-quad (rewards sum, terminated OR, export after the quad)."""
    out = []
    for q in range(len(trace) // 4):
        rew = np.zeros((n, 4), np.float32)
        term = np.zeros(n, np.uint8)
        for k in range(4):
            ref.step(trace[4 * q + k].cpu().numpy(), autoreset=True)
            e = ref.export()
            rew += e["rewards"]
            term |= e["terminated"]
        out.append((rew, term, e))
    return out


def test_roll_out_and_gae_match_oracle_replay():
    """src/roll_out.py:49-108 + src/gae.py with the ppo.py defaults (T scaled down)."""
    from brl_b200.gae import make_calc_gae
    from brl_b200.models import init_params, make_forward_pass, params_to_numpy
    from brl_b200.roll_out import make_roll_out
    from brl_b200 import random as brandom
    from oracle import oracle as orc
    env, table = _mk_env()
    n, T = 512, 12
    config = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, game_mode="competitive",
                  num_steps=T, reward_scale=7600.0, gamma=1.0, gae_lambda=0.95)
    fp = make_forward_pass("relu", "DeepMind")
    params, opp_params = init_params(1, DEV), init_params(2, DEV)
    keys = env.make_keys(77, n)
    state = env.init(keys)
    runner = (params, None, state, state.observation, torch.zeros((), dtype=torch.int64, device=DEV), brandom.PRNGKey(3))
    roll_out = make_roll_out(config, env, fp, fp)
    trace = []
    runner2, traj = roll_out(runner, opp_params, trace=trace)
    assert len(trace) == 4 * T
    ref = orc.OracleEnv(table, n)
    ref.init(keys.cpu().numpy().view(np.uint64))
    e0 = ref.export()
    assert (traj.obs[0].float().cpu().numpy() == e0["observation"]).all()   # recorded in the policy's input dtype (bf16 0/1)
    actor = e0["current_player"].copy()
    quads = _replay_quads(ref, trace, n)
    np_params = params_to_numpy(params)
    n_term = 0
    for t, (rew, term, e) in enumerate(quads):
        assert (traj.action[t].cpu().numpy() == trace[4 * t].cpu().numpy()).all()
        assert (traj.done[t].cpu().numpy() == term.astype(bool)).all(), f"done t={t}"
        want_r = rew[np.arange(n), actor] / np.float32(7600.0)
        assert (traj.reward[t].cpu().numpy() == want_r).all(), f"reward t={t}"
        obs_next = traj.obs[t + 1] if t + 1 < T else runner2[3]
        assert (obs_next.float().cpu().numpy() == e["observation"]).all(), f"obs t={t}"
        if t + 1 < T:
            assert (traj.legal_action_mask[t + 1].cpu().numpy() == e["legal_action_mask"].astype(bool)).all()
        # the recorded action was legal and its log-prob is the masked log-softmax of the actor's logits
        logits, value = orc.mlp_forward(np_params, traj.obs[t].float().cpu().numpy())
        mask_t = traj.legal_action_mask[t].cpu().numpy()
        a = traj.action[t].cpu().numpy()
        assert mask_t[np.arange(n), a].all()
        ml = np.where(mask_t, logits.astype(np.float64), -np.inf)
        lse = np.log(np.exp(ml - ml.max(1, keepdims=True)).sum(1)) + ml.max(1)
        np.testing.assert_allclose(traj.log_prob[t].cpu().numpy(), ml[np.arange(n), a] - lse, rtol=2e-4, atol=2e-4)
        np.testing.assert_allclose(traj.value[t].cpu().numpy(), value, rtol=2e-4, atol=2e-4)
        actor = e["current_player"].copy()
        n_term += int(term.sum())
    assert int(runner2[4]) == n_term and n_term > 0
    # GAE on the recorded trajectory (bootstrap value from the last observation, src/gae.py:16-18)
    calc_gae = make_calc_gae(config, fp)
    adv, tgt = calc_gae(runner2, traj)
    _, last_val = fp.apply(params, runner2[3])
    adv_ref, tgt_ref = orc.gae(traj.done.cpu().numpy().astype(np.uint8), traj.value.cpu().numpy(), traj.reward.cpu().numpy(),
                               last_val.cpu().numpy(), 1.0, 0.95)
    np.testing.assert_allclose(adv.cpu().numpy(), adv_ref, rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(tgt.cpu().numpy(), tgt_ref, rtol=1e-6, atol=1e-7)


def test_roll_out_cuda_graph_replay_equals_traced_launches():
    """From 4096 envs on the T-step rollout is ONE CUDA graph replay.  With the same seeding scheme the plain-launch path
    (traced and replayed through the oracle env) must give the bit-identical trajectory, and a second replay must draw
    fresh noise (the per-rollout key is a device word, not a captured constant)."""
    from brl_b200.models import init_params, make_forward_pass
    from brl_b200.roll_out import make_roll_out
    from brl_b200 import random as brandom
    from oracle import oracle as orc
    env, table = _mk_env()
    n, T = 4096, 5
    config = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, game_mode="competitive",
                  num_steps=T, reward_scale=7600.0, gamma=1.0, gae_lambda=0.95)
    params, opp_params = init_params(1, DEV), init_params(2, DEV)
    keys = env.make_keys(78, n)

    def fresh_runner():
        state = env.init(keys)
        return (params, None, state, state.observation, torch.zeros((), dtype=torch.int64, device=DEV), brandom.PRNGKey(9))

    fp_g = make_forward_pass("relu", "DeepMind")
    roll_g = make_roll_out(config, env, fp_g, fp_g)
    runner_g, traj_g = roll_g(fresh_runner(), opp_params)                    # captures, then replays
    got = {k: getattr(traj_g, k).clone() for k in traj_g._fields}
    last_obs_g, count_g = runner_g[3].clone(), int(runner_g[4])
    fp_e = make_forward_pass("relu", "DeepMind")
    roll_e = make_roll_out(config, env, fp_e, fp_e)
    trace = []
    runner_e, traj_e = roll_e(fresh_runner(), opp_params, trace=trace, graph_seeding=True)
    for k in traj_e._fields:
        assert torch.equal(got[k], getattr(traj_e, k)), k
    assert torch.equal(last_obs_g, runner_e[3]) and count_g == int(runner_e[4]) and runner_g[5] == runner_e[5]
    # the traced run is a faithful rollout of the oracle env
    ref = orc.OracleEnv(table, n)
    ref.init(keys.cpu().numpy().view(np.uint64))
    actor = ref.export()["current_player"].copy()
    n_term = 0
    for t, (rew, term, e) in enumerate(_replay_quads(ref, trace, n)):
        assert (traj_e.done[t].cpu().numpy() == term.astype(bool)).all()
        assert (traj_e.reward[t].cpu().numpy() == rew[np.arange(n), actor] / np.float32(7600.0)).all()
        actor = e["current_player"].copy()
        n_term += int(term.sum())
    assert count_g == n_term
    # second replay from the SAME start state: different per-rollout key -> different samples
    _, traj_g2 = roll_g(fresh_runner()[:5] + (brandom.PRNGKey(10),), opp_params)
    assert not torch.equal(traj_g2.action, got["action"])
    # and continuing from the returned runner state works without copies going wrong (state aliases the graph's buffers)
    runner_g3, traj_g3 = roll_g(runner_g, opp_params)
    assert int(runner_g3[4]) >= count_g and torch.isfinite(traj_g3.value).all()


@pytest.mark.parametrize("mode", ["deterministic", "free-run"])
def test_quad_step_variants_match_oracle_replay(mode):
    """src/utils.py:133-246 without auto-reset (the evaluation loops' use)."""
    from brl_b200 import utils
    from brl_b200.models import init_params, make_forward_pass
    from brl_b200 import random as brandom
    from oracle import oracle as orc
    env, table = _mk_env()
    n = 256
    fp = make_forward_pass("relu", "DeepMind")
    pa, pb = init_params(5, DEV), init_params(6, DEV)
    make = (utils.single_play_step_two_policy_commpetitive_deterministic if mode == "deterministic"
            else utils.single_play_step_free_run)
    step_fn = make(step_fn=env.step, actor_forward_pass=fp, actor_params=pa, opp_forward_pass=fp, opp_params=pb)
    step_fn.trace = trace = []
    keys = env.make_keys(9, n)
    state = env.init(keys)
    ref = orc.OracleEnv(table, n)
    ref.init(keys.cpu().numpy().view(np.uint64))
    rng = brandom.PRNGKey(1)
    for it in range(6):
        action = torch.as_tensor(ref.random_legal_actions(4, it), device=DEV)
        state = step_fn(state, action, rng)
        rew, term = np.zeros((n, 4), np.float32), np.zeros(n, np.uint8)
        for k in range(4):
            a = trace[4 * it + k].cpu().numpy()
            if mode == "free-run" and k in (1, 3):
                assert (a == 0).all()  # opponents always pass
            ref.step(a)
            e = ref.export()
            rew += e["rewards"]
            term |= e["terminated"]
        assert (state.rewards.cpu().numpy() == rew).all()
        assert (state.terminated.cpu().numpy() == term.astype(bool)).all()
        assert (state.observation.cpu().numpy() == e["observation"]).all()
        assert (state.legal_action_mask.cpu().numpy() == e["legal_action_mask"].astype(bool)).all()


def test_simple_duplicate_evaluate_matches_oracle_replay():
    """eval.py / src/evaluation.py:69-204 on the 1000 real boards' table, 100 envs."""
    from brl_b200 import BridgeBidding
    from brl_b200.evaluation import make_simple_duplicate_evaluate
    from brl_b200.models import init_params, params_to_numpy
    from brl_b200 import random as brandom
    from oracle import oracle as orc
    boards = H.load_boards()
    env = BridgeBidding(table=boards["table"], device=DEV)
    n = 100  # eval.py:28 num_eval_envs
    p1, p2 = init_params(11, DEV), init_params(12, DEV)
    evaluate = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n)
    trace = []
    rng = brandom.PRNGKey(0)
    (mean, se, win), info_a, info_b, cum = evaluate(p1, p2, rng, trace=trace)
    _, sub = brandom.split(rng)
    keys = env.make_keys(sub, n).cpu().numpy().view(np.uint64)
    ref = orc.OracleEnv(boards["table"], n)
    ref.init(keys)
    ref.duplicate_tables_from_state()
    cum_ref = np.zeros(n)
    np1, np2 = params_to_numpy(p1), params_to_numpy(p2)
    agree = total = 0
    for action, l1, l2 in trace:
        e = ref.export()
        live = e["terminated"] == 0
        # action choice: NumPy MLP + masked argmax on the oracle's observation
        lg1, _ = orc.mlp_forward(np1, e["observation"])
        lg2, _ = orc.mlp_forward(np2, e["observation"])
        lg = np.where((e["current_player"] < 2)[:, None], lg1, lg2)
        want, _ = orc.categorical(lg, e["legal_action_mask"], sample=False)
        got = action.cpu().numpy()
        agree += int((want[live] == got[live]).sum())
        total += int(live.sum())
        ref.duplicate_step(got)
        cum_ref += ref.export()["rewards"][:, 0]
    assert ref.export()["terminated"].all()
    assert (cum.cpu().numpy() == cum_ref).all()
    assert agree / total > 0.995, f"argmax agreement {agree}/{total} (near-ties flip between cuBLAS and NumPy summation order)"
    # each net ran only on the live envs its team decides (src/evaluation.py:124-151 runs both nets on all n every iteration)
    assert evaluate.rows_forwarded == total and total < len(trace) * n
    want_stats = orc.match_stats(cum_ref)
    np.testing.assert_allclose([mean, se, win], want_stats, rtol=1e-9, atol=1e-12)
    for buf, info in ((info_a, ref.info_a), (info_b, ref.info_b)):
        assert (buf.terminated.cpu().numpy() == info["terminated"]).all()
        assert (buf.rewards.cpu().numpy() == info["rewards"]).all()
        assert (buf.last_bid.cpu().numpy() == info["last_bid"]).all()
        assert (buf.last_bidder.cpu().numpy() == info["last_bidder"]).all()


def test_simple_evaluate_matches_oracle_replay():
    """src/evaluation.py:11-66 (the per-iteration strength probe of ppo.py:366): deterministic quad steps against a
    fixed opponent on the 1000 real boards; the traced sub-step actions are replayed on the oracle and the per-env
    return R = sum of rewards[actor] must be bit-equal, R.mean() equal, and the GPU's argmax decisions must be the
    float64 NumPy MLP's wherever they are not near-ties."""
    from brl_b200 import BridgeBidding
    from brl_b200.evaluation import make_simple_evaluate
    from brl_b200.models import init_params, params_to_numpy
    from brl_b200 import random as brandom
    from oracle import oracle as orc
    boards = H.load_boards()
    env = BridgeBidding(table=boards["table"], device=DEV)
    n = 128
    p_actor, p_opp = init_params(4, DEV), init_params(3, DEV)
    ev = make_simple_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", None, n, team2_params=p_opp)
    trace = []
    rng = brandom.PRNGKey(5)
    mean = ev(p_actor, rng, trace=trace)
    tag, R = trace.pop()
    assert tag == "R" and len(trace) % 4 == 0
    _, sub = brandom.split(rng)
    ref = orc.OracleEnv(boards["table"], n)
    ref.init(env.make_keys(sub, n).cpu().numpy().view(np.uint64))
    np_actor, np_opp = params_to_numpy(p_actor), params_to_numpy(p_opp)
    R_ref = np.zeros(n, np.float32)
    agree = total = 0
    for it in range(len(trace) // 4):
        actor = ref.export()["current_player"].astype(np.int64)
        rew = np.zeros((n, 4), np.float32)
        for k in range(4):
            e = ref.export()
            live = e["terminated"] == 0
            got = trace[4 * it + k].cpu().numpy()
            lg, _ = orc.mlp_forward(np_opp if k in (1, 3) else np_actor, e["observation"])   # src/utils.py:150-196
            want, _ = orc.categorical(lg, e["legal_action_mask"], sample=False)
            agree += int((want[live] == got[live]).sum())
            total += int(live.sum())
            ref.step(got)                                # a finished env: zero-reward no-op (src/evaluation.py:31-33)
            rew += ref.export()["rewards"]
        R_ref += rew[np.arange(n), actor]                                                    # src/evaluation.py:58
    assert ref.export()["terminated"].all()
    assert (R.cpu().numpy() == R_ref).all()
    assert abs(float(mean) - float(R_ref.astype(np.float64).mean())) <= 1e-6 * max(1.0, abs(float(R_ref.mean())))
    assert np.abs(R_ref).max() <= 7600 and (R_ref != 0).any()
    assert agree / total > 0.995, f"argmax agreement {agree}/{total}"


def test_league_evaluate_equals_separate_matches():
    """configs[4] host logic: block m of the global env range plays pool model m; identical to running the
    matches one by one on the same global indices (so the result cannot depend on how ranks shard it)."""
    from brl_b200 import BridgeBidding
    from brl_b200.evaluation import make_league_evaluate, make_simple_duplicate_evaluate
    from brl_b200.models import init_params
    from brl_b200 import random as brandom
    env, _ = _mk_env()
    n_total, n_models = 600, 3
    actor = init_params(41, DEV)
    pool = [init_params(50 + m, DEV) for m in range(n_models)]
    league = make_league_evaluate(env, "relu", "DeepMind", n_total, n_models)
    rng = brandom.PRNGKey(2)
    res = league(actor, pool, rng)
    assert len(res) == n_models
    for m in range(n_models):
        single = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", 200, env_offset=200 * m)
        (mean, se, win), _, _, _ = single(actor, pool[m], rng)
        np.testing.assert_allclose(res[m], (mean, se, win), rtol=1e-12)
    assert len({round(r[0], 6) for r in res}) == n_models  # three different opponents, three different results


def test_c1_eval_match_with_seeded_weights_reproduces_golden():
    """BASELINE configs[0] / eval.py:43-65 (num_eval_envs=100, the 1000 real boards) played by two seeded nets of the
    bundled models' architecture (tests/helpers.seeded_params) on the GPU path (tensor-core forward, duplicate_step
    kernel).  Every live decision must equal the frozen float64 decision (the smallest top-2 gap of the match is 3.7e-3,
    far above the forward's 1e-5 error), and IMP mean +- SE, the per-board IMPs and both tables' contracts must equal
    the golden values, which the reference's own scorer reproduced (tests/golden/make_c1_golden.py --seeded)."""
    from brl_b200 import BridgeBidding
    from brl_b200.evaluation import make_simple_duplicate_evaluate
    from brl_b200 import random as brandom
    g = H.load_c1_seeded()
    boards = H.load_boards()
    env = BridgeBidding(table=boards["table"], device=DEV)
    n = int(g["n"])
    p1, p2 = (H.seeded_params(int(s), DEV) for s in g["weight_seeds"])
    evaluate = make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n)
    trace = []
    (mean, se, win), info_a, info_b, cum = evaluate(p1, p2, brandom.PRNGKey(int(g["seed"])), trace=trace)
    steps = g["actions"].shape[0]
    assert len(trace) >= steps
    for t in range(steps):
        live = g["live"][t] != 0
        got = trace[t][0].cpu().numpy()
        assert (got[live] == g["actions"][t][live]).all(), f"step {t}: decisions differ from the float64 golden ones"
    assert (cum.cpu().numpy() == g["imps"]).all()
    np.testing.assert_allclose([mean, se, win], g["stats"], rtol=1e-9, atol=1e-12)
    for k, info in (("a", info_a), ("b", info_b)):
        assert (info.last_bid.cpu().numpy() == g[k + "_last_bid"]).all()
        assert (info.last_bidder.cpu().numpy() == g[k + "_last_bidder"]).all()
        assert (info.rewards.cpu().numpy() == g[k + "_rewards"]).all()


def test_empty_batch_is_a_no_op_for_every_batched_op():
    """n_envs = 0 (an empty shard, a zero-size XLA / torch buffer whose pointer is NULL): every batched op returns BRL_OK
    without requiring or touching its buffers; brl_team_rows still reports two empty lists."""
    import ctypes as C
    from brl_b200 import _lib
    L = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    nulls = (C.c_void_p * 24)()
    p0 = _lib.BrlParams(0, 0, 0, 1, 10, _lib.F_AUTORESET, 0, 4, -1.0, 1.0, 0.99, 0.95)
    for name in ("brl_make_keys", "brl_init", "brl_reset_fields", "brl_step", "brl_duplicate_init", "brl_duplicate_step", "brl_observe",
                 "brl_legal_mask", "brl_rollout_random", "brl_state_fields", "brl_gae", "brl_categorical", "brl_imp_reward",
                 "brl_match_stats", "brl_gather_reward", "brl_obs_to_bf16", "brl_mlp_forward", "brl_policy_act", "brl_policy_act_rows",
                 "brl_gather_rows", "brl_eval_act_log", "brl_eval_summary"):
        rc = getattr(L, name)(C.c_void_p(stream), nulls, C.byref(p0), C.sizeof(p0))
        assert rc == 0, (name, L.brl_last_error())
    counts = torch.full((2,), 7, dtype=torch.int32, device=DEV)
    bufs = (C.c_void_p * 5)(None, None, None, None, counts.data_ptr())
    assert L.brl_team_rows(C.c_void_p(stream), bufs, C.byref(p0), C.sizeof(p0)) == 0
    assert counts.tolist() == [0, 0]
    # ... and a non-empty call with a NULL required buffer is still an error, not a crash
    p1 = _lib.BrlParams(8, 0, 8, 1, 10, 0, 0, 0, -1.0, 1.0, 0.0, 0.0)
    assert L.brl_step(C.c_void_p(stream), nulls, C.byref(p1), C.sizeof(p1)) == -2
    assert b"NULL" in L.brl_last_error()
