"""GPU: the model zoo packed in HBM and the PFSP probe as one league call -- the probe bit-equals a duplicate match per zoo
model (device loop and host loop), the zoo's slots hold what was appended in the host list's order, a chosen opponent
survives the ring reusing its slot, a packed opponent drives the rollout exactly as its fp32 parameters do, and ppo.train
with the device zoo equals the host zoo, including its up-front fallback."""
import numpy as np
import pytest
import torch

from tests import helpers as H

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
_NETS = {}


def _net(seed):
    if seed not in _NETS:
        _NETS[seed] = H.seeded_params(seed, DEV)
    return _NETS[seed]


def _env(rows=3000, seed=6):
    from brl_b200 import BridgeBidding
    from brl_b200.deals import synthetic_deal_table
    return BridgeBidding(table=synthetic_deal_table(rows, seed=seed), device=DEV)


def _pack(params):
    from brl_b200 import ops
    from brl_b200.models import LAYERS
    return ops.mlp_pack([params[k]["w"] for k in LAYERS], [params[k]["b"] for k in LAYERS])


PROBES = [(K, n, p, 1 << 20) for K in (1, 3, 17) for n in (1, 100, 257) for p in ("tc", "tc-bf16")] + \
         [(17, 100, "tc", 300), (17, 257, "tc-bf16", 600), (3, 100, "tc", 100)]   # several chunks


@pytest.mark.parametrize("case", range(len(PROBES)))
def test_probe_equals_one_duplicate_match_per_zoo_model(case, monkeypatch):
    import brl_b200.evaluation as ev
    from brl_b200 import random as brandom
    from brl_b200.zoo import ModelZoo
    K, n, precision, max_envs = PROBES[case]
    orig = ev.make_forward_pass
    monkeypatch.setattr(ev, "make_forward_pass", lambda **kw: orig(precision=precision, **kw))
    env = _env()
    current = _net(800)
    zoo = ModelZoo(K, DEV)
    for k in range(K + 2):                                   # the ring wraps: logical order is not slot order
        zoo.append(_net(810 + k))
    models = [_net(810 + k) for k in range(2, K + 2)]
    key = brandom.PRNGKey(40 + case)
    got_ret = {}
    got = ev.make_device_pfsp_probe(env, "relu", "DeepMind", n, max_envs=max_envs)(current, zoo, key, cum_returns=got_ret)
    assert len(got) == K and sorted(got_ret) == list(range(K))
    device_match = ev.make_device_duplicate_evaluate(env, "relu", "DeepMind", n)
    host_match = ev.make_simple_duplicate_evaluate(env, "relu", "DeepMind", "relu", "DeepMind", n)
    for k, model in enumerate(models):
        d_log, _, _, d_ret = device_match(current, model, key)
        h_log, _, _, h_ret = host_match(current, model, key)
        assert torch.equal(got_ret[k], d_ret) and torch.equal(got_ret[k], h_ret), k
        np.testing.assert_array_equal(got[k], d_log, err_msg=str(k))   # integer IMP sums: the same numbers (SE: nan at n = 1)
        np.testing.assert_array_equal(got[k], h_log, err_msg=str(k))


def test_zoo_slots_hold_the_appended_models_in_host_order():
    from brl_b200.zoo import ModelZoo
    for capacity in (1, 3):
        zoo, host = ModelZoo(capacity, DEV), []
        for s in range(820, 827):
            zoo.append(_net(s))
            host.append(s)
            host[:] = host[-capacity:]
            assert len(zoo) == len(host)
            for k, seed in enumerate(host):
                assert torch.equal(zoo.blob(zoo.slot(k)), _pack(_net(seed))), (capacity, s, k)
            assert not zoo.pool[:, zoo.blob(0).numel():].any()      # pool padding stays zero


def test_opponent_is_unchanged_after_its_slot_is_reused():
    from brl_b200.zoo import ModelZoo
    zoo = ModelZoo(2, DEV)
    zoo.append(_net(830))
    zoo.append(_net(831))
    opp, slot = zoo.opponent(0), zoo.slot(0)
    zoo.append(_net(832))
    zoo.append(_net(833))
    assert torch.equal(zoo.blob(slot), _pack(_net(832)))
    assert torch.equal(opp.blob, _pack(_net(830)))


@pytest.mark.parametrize("graph", [True, False])
def test_rollout_with_a_packed_opponent_equals_fp32_params(graph, monkeypatch):
    from brl_b200 import random as brandom
    from brl_b200.models import PackedParams, make_forward_pass
    from brl_b200.roll_out import make_roll_out
    if not graph:
        monkeypatch.setenv("BRL_ROLLOUT_GRAPH", "0")
    env = _env(5000, seed=8)
    n, T = 4096, 4
    config = dict(actor_illegal_action_mask=True, actor_illegal_action_penalty=False, game_mode="competitive",
                  num_steps=T, reward_scale=7600.0)
    params, opp = _net(840), _net(841)
    keys = env.make_keys(91, n)
    fp = make_forward_pass("relu", "DeepMind")
    roll_out = make_roll_out(config, env, fp, fp)
    out = []
    for opp_params in (opp, PackedParams(_pack(opp)), opp):
        state = env.init(keys)
        runner = (params, None, state, state.observation, torch.zeros((), dtype=torch.int64, device=DEV), brandom.PRNGKey(5))
        runner, traj = roll_out(runner, opp_params)
        out.append(([getattr(traj, k).clone() for k in traj._fields], runner[3].clone(), int(runner[4]), runner[5]))
    for other in out[1:]:
        assert all(torch.equal(a, b) for a, b in zip(out[0][0], other[0]))
        assert torch.equal(out[0][1], other[1]) and out[0][2:] == other[2:]


def _train(prioritized, zoo_size):
    from brl_b200 import ppo, random as brandom
    from brl_b200.deals import synthetic_deal_table
    config = dict(num_envs=4096, num_steps=2, minibatch_size=2048, update_epochs=1, total_timesteps=4096 * 2 * 6,
                  num_eval_envs=512, num_prioritized_envs=100, num_eval_step=3, self_play=True, ratio_model_zoo=1.0,
                  num_model_zoo=zoo_size, save_model_interval=1, prioritized_fictitious=prioritized, lr=1e-4, save_model=False)
    return ppo.train(config, brandom.PRNGKey(2), tables=[synthetic_deal_table(300, seed=k) for k in range(2)],
                     eval_table=synthetic_deal_table(400, seed=9), device=DEV, eval_opp_params=_net(850))


def _assert_same_run(a, b):
    from brl_b200.models import params_to_numpy
    (runner_a, logs_a), (runner_b, logs_b) = a, b
    assert len(logs_a) == len(logs_b) == 6
    for la, lb in zip(logs_a, logs_b):
        keys = sorted(k for k in la if k.startswith(("train/", "eval/")) or k in ("board_num", "steps", "table"))
        assert keys == sorted(k for k in lb if k.startswith(("train/", "eval/")) or k in ("board_num", "steps", "table"))
        for k in keys:
            np.testing.assert_allclose(lb[k], la[k], rtol=1e-12, atol=0, err_msg=k)
    pa, pb = params_to_numpy(runner_a[0]), params_to_numpy(runner_b[0])
    assert all((pa[k] == pb[k]).all() for k in pa)


@pytest.mark.parametrize("zoo_size", [1, 2])
@pytest.mark.parametrize("prioritized", [True, False])
def test_ppo_train_with_the_device_zoo_equals_the_host_list_zoo(prioritized, zoo_size, monkeypatch):
    """six iterations, a save every iteration and a one- or two-model zoo, so the ring wraps; the runs contain an append that
    reuses the slot of the opponent chosen in the iteration before, which that iteration's imp_opp probe still plays.  The
    reference run plays the host loops with the host-list zoo.  Then the same run with the device zoo refused by the memory
    budget."""
    import brl_b200.ppo as ppo
    from brl_b200.zoo import ModelZoo
    made, events = [], []

    class RecordedZoo(ModelZoo):
        def __init__(self, *a):
            super().__init__(*a)
            made.append(self)

        def append(self, params):
            evicted = self.slot(0) if len(self) == self.capacity else None
            super().append(params)
            events.append(("append", evicted))

        def opponent(self, k):
            events.append(("opponent", self.slot(k)))
            return super().opponent(k)
    monkeypatch.setattr(ppo, "ModelZoo", RecordedZoo)
    probes = []
    orig_probe = ppo.make_device_pfsp_probe

    def counting_probe(*a, **kw):
        probe = orig_probe(*a, **kw)

        def counted(*pa, **pkw):
            probes.append(1)
            return probe(*pa, **pkw)
        counted.reserve = probe.reserve
        return counted
    monkeypatch.setattr(ppo, "make_device_pfsp_probe", counting_probe)
    with monkeypatch.context() as m:   # the host loops, with the host-list zoo and its one match per model
        m.setattr(ppo, "make_evaluators", H.host_evaluators)
        m.setattr(ppo, "device_zoo_fits", lambda *a, **kw: False)
        host = _train(prioritized, zoo_size)
    assert not made
    device = _train(prioritized, zoo_size)
    assert len(made) == 1 and made[0].capacity == zoo_size and len(made[0]) == zoo_size
    assert len(probes) == (5 if prioritized else 0)                    # one call per PFSP draw (iterations 1..5)
    assert [e for e in events if e[0] == "opponent"]
    if zoo_size == 1 or not prioritized:   # certain with one model; FSP's seeded uniform draws hit it with two.  PFSP picks
        # the newest of two models in every iteration of this run, so there the slot reused is never the opponent's
        assert any(a[0] == "opponent" and b == ("append", a[1]) for a, b in zip(events, events[1:])), events
    _assert_same_run(host, device)
    free, total = torch.cuda.mem_get_info(DEV)
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (1 << 30, total))
    fallback = _train(prioritized, zoo_size)
    assert len(made) == 1 and len(probes) == (5 if prioritized else 0)
    _assert_same_run(host, fallback)
