"""Counterfactual call values (DESIGN.md f16) in plain Python: the one reference for brl_call_values.  Restates the
definitions next to `call_value_gain` in csrc/env_device.cuh:

  base match   the duplicate match brl_duplicate_match plays for the same keys, pool and env_models (masked argmax)
  decision d   a step where the env is live at table T (A or B): pre-step state S_d, player p to act, its net m
               (brl_model_rows' rule), context c = system_context (tests/system_ref.py), played call b_d
  branch (d,a) for every call a legal in S_d: step S_d with a (no auto-reset, no table switch), play that one table to its end
               with every player's own net (masked argmax); r_d(a) = the branch's final rewards[0] (NaN: a illegal)
  gain         g_d(a) = sigma_p * (imp(r_d(a) + R_other) - imp(R_A + R_B)), sigma_p = +1 for players 0/1, -1 for 2/3
  regret       regret_d = max over legal a of g_d(a) >= 0
  invariant    r_d(b_d) = R_T (the played branch is the base game)
  sums         gain_sums[m, c, b, a] += {1, g, g^2, g > 0}; regret_sums[m, c] += {1, regret, regret^2, regret > 0};
               mismatch[m] += r_d(b_d) != R_T"""
import numpy as np

CONTEXTS, NUM_ACTIONS = 75, 38
IMP_THRESHOLDS = (20, 50, 90, 130, 170, 220, 270, 320, 370, 430, 500, 600, 750, 900, 1100, 1300, 1500, 1750, 2000, 2250,
                  2500, 3000, 3500, 4000)


def imp(d: float) -> int:
    """the IMPs of a point difference d (src/duplicate.py:46-69: thresholds reached by |d|, signed by d >= 0)"""
    k = sum(abs(d) >= t for t in IMP_THRESHOLDS)
    return k if d >= 0 else -k


def gains(r, R_a: float, R_b: float, table: int, player: int):
    """g_d(a) for the 38 calls (None where r is NaN: an illegal call) of a decision at `table` (0 A, 1 B) by `player`"""
    other = R_b if table == 0 else R_a
    base = imp(R_a + R_b)
    sign = 1 if player < 2 else -1
    return [None if np.isnan(x) else sign * (imp(float(x) + other) - base) for x in r]


def regret(g) -> int:
    return max(x for x in g if x is not None)


def new_sums(n_models: int):
    return (np.zeros((n_models, CONTEXTS, NUM_ACTIONS, NUM_ACTIONS, 4), np.int64), np.zeros((n_models, CONTEXTS, 4), np.int64),
            np.zeros(n_models, np.int64))


def reduce_records(rec, R_a, R_b, n_models: int):
    """(gain_sums, regret_sums, mismatch) of decision records: rec holds arrays env, table, player, net, context, played and
    r[., 38]; R_a / R_b are the base results by env"""
    gain, reg, mismatch = new_sums(n_models)
    for k in range(len(rec["env"])):
        e, t, p, m, c, b = (int(rec[f][k]) for f in ("env", "table", "player", "net", "context", "played"))
        g = gains(rec["r"][k], float(R_a[e]), float(R_b[e]), t, p)
        for a, x in enumerate(g):
            if x is not None:
                gain[m, c, b, a] += (1, x, x * x, int(x > 0))
        rg = regret(g)
        reg[m, c] += (1, rg, rg * rg, int(rg > 0))
        mismatch[m] += float(rec["r"][k][b]) != float(R_b[e] if t else R_a[e])
    return gain, reg, mismatch


def host_records(env, nets, models, n, rng_key, precision="tc", tune=0):
    """The decision records of the host loop: make_simple_duplicate_evaluate's match (record=) gives the played calls, its
    per-step states are replayed with ops.duplicate_step, every legal call of every live env is stepped with ops.step, and
    each branch continues with ops.policy_act_rows per net until done.  `models` = (i, j) by team or (a, b, c, d) by player.
    Returns (records, R_a, R_b) with records' env = the env index."""
    import torch
    from brl_b200 import ops, random as brandom
    from brl_b200 import evaluation as ev
    from brl_b200.duplicate import Table_info, duplicate_step
    from brl_b200.models import make_forward_pass
    from tests import system_ref
    dev = env.device
    fp = make_forward_pass("relu", "DeepMind", precision=precision)
    single = precision == "tc-bf16"
    by_player = list(models) if len(models) == 4 else [models[0], models[0], models[1], models[1]]
    host = ev.make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n)
    record = []
    orig = ops.policy_act_rows  # the host loop's forwards take `precision` and `tune`
    ops.policy_act_rows = lambda *a, **kw: orig(*a, **{**kw, "tune": kw.get("tune", 0) | tune, "single_bf16": single})
    try:
        kw = {} if len(models) == 2 else dict(team1_partner=nets[models[1]], team2_partner=nets[models[3]])
        a, b = (models[0], models[1]) if len(models) == 2 else (models[0], models[2])
        _, ta, tb, _ = host(nets[a], nets[b], rng_key, record=record, **kw)
    finally:
        ops.policy_act_rows = orig
    R_a, R_b = ta.rewards[:, 0].cpu().numpy(), tb.rewards[:, 0].cpu().numpy()
    _, sub = brandom.split(rng_key)
    state = ev._bf16_state(env, env.make_keys(sub, n))
    tinfo = [Table_info.from_state(state), Table_info.from_state(state)]
    step_fn = duplicate_step(env.step)
    rec = {f: [] for f in ("env", "table", "player", "net", "context", "played", "r")}
    packed_blobs = [fp._packed(p) for p in nets]
    for action, a_done, _ in record:
        live = np.flatnonzero(state._terminated_u8.cpu().numpy() == 0)
        mask = state._mask_u8.cpu().numpy().astype(bool)
        player = state.current_player.cpu().numpy()
        pairs = [(i, c) for i in live for c in np.flatnonzero(mask[i])]
        r = np.full((len(live), NUM_ACTIONS), np.nan, np.float32)
        if pairs:
            idx = torch.as_tensor([i for i, _ in pairs], device=dev)
            B = len(pairs)
            packed = state._packed[:, idx, :].contiguous()
            out = ops.EnvOutputs(B, dev, torch.bfloat16)
            act = torch.as_tensor([c for _, c in pairs], dtype=torch.int32, device=dev)
            ops.step(packed, act, env.table, packed, out)
            val = out.rewards[:, 0].clone()
            nets_of = torch.as_tensor(np.array(by_player, np.int64), device=dev)
            scratch = torch.empty(ops._lib.load().brl_mlp_rows_scratch_bytes(B), dtype=torch.uint8, device=dev)
            for _ in range(320):
                done = out.terminated.bool()
                if bool(done.all()):
                    break
                net = nets_of[out.current_player.long()]
                for m in range(len(nets)):
                    rows = torch.nonzero(~done & (net == m)).flatten().to(torch.int32)
                    if rows.numel():
                        ops.policy_act_rows(out.observation, packed_blobs[m], scratch, out.legal_action_mask, act, rows,
                                            single_bf16=single, tune=tune)
                ops.step(packed, act, env.table, packed, out)
                val += out.rewards[:, 0]
            pos = {i: k for k, i in enumerate(live)}
            for (i, c), v in zip(pairs, val.cpu().numpy()):
                r[pos[i], c] = v
        act_h = action.numpy()
        for k, i in enumerate(live):
            p = int(player[i])
            rec["env"].append(i)
            rec["table"].append(int(a_done[i] != 0))
            rec["player"].append(p)
            rec["net"].append(by_player[p])
            rec["played"].append(int(act_h[i]))
            rec["r"].append(r[k])
        state, tinfo[0], tinfo[1] = step_fn(state, action.to(dev), tinfo[0], tinfo[1])
    # contexts from each table's call sequence (tests/system_ref.py's reader)
    calls = {}
    for k, (e, t) in enumerate(zip(rec["env"], rec["table"])):
        seq = calls.setdefault((e, t), [])
        seq.append(rec["played"][k])
        rec["context"].append(system_ref.context(seq, len(seq) - 1))
    out = {f: np.asarray(v, np.float32 if f == "r" else np.int32) for f, v in rec.items()}
    out["r"] = out["r"].reshape(-1, NUM_ACTIONS)
    return out, R_a, R_b
