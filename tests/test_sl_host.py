"""Supervised pre-training on the host: the data-file parser (sl.py:87-97), the deal packing, the C oracle's replay of
stored auction prefixes against the reference's own examples (tests/golden/make_sl_golden.py), the trajectory stream,
and hand-worked answers of the float64 restatement oracle/sl_ref.py."""
import os

import numpy as np
import pytest
import torch

from tests.helpers import GOLDEN


def _golden():
    z = np.load(os.path.join(GOLDEN, "sl_golden.npz"))
    return {k: z[k] for k in z.files}


def _write(tmp_path, lines):
    p = tmp_path / "data.txt"
    p.write_text("\n".join(lines) + "\n")
    return str(p)


def _deal(seed=0):
    return [int(x) for x in np.random.default_rng(seed).permutation(52)]


def test_parser_keeps_passed_out_lines_whole_and_strips_play_tails(tmp_path):
    from brl_b200 import sl
    d0, d1 = _deal(0), _deal(1)
    auction = [52 + 3, 52 + 0, 52 + 0, 52 + 0]         # 1C P P P
    tail = _deal(2)
    path = _write(tmp_path, [" ".join(map(str, d0 + [52] * 4)), "", " ".join(map(str, d1 + auction + tail))])
    t = sl.parse_trajectories(path)
    assert len(t) == 2
    assert t.offsets.tolist() == [0, 4, 8]
    assert t.calls.tolist() == [0, 0, 0, 0, 3, 0, 0, 0]
    assert t.line.tolist() == [1, 3]                  # the blank line is skipped, numbering follows the file


@pytest.mark.parametrize("bad,msg", [
    ("deal", "not a permutation"),
    ("call", "outside 52..89"),
    ("short", "no call"),
    ("token", "not an integer"),
])
def test_parser_rejects_bad_lines_with_their_line_number(tmp_path, bad, msg):
    from brl_b200 import sl
    good = " ".join(map(str, _deal(0) + [52] * 4))
    if bad == "deal":
        d = _deal(1)
        d[5] = d[6]
        line = " ".join(map(str, d + [52] * 4))
    elif bad == "call":
        line = " ".join(map(str, _deal(1) + [55, 52, 90, 52] + _deal(2)))
    elif bad == "short":
        line = " ".join(map(str, _deal(1) + [52] * 3))
    else:
        line = " ".join(map(str, _deal(1) + [52] * 3)) + " x"
    path = _write(tmp_path, [good, good, line, good])
    with pytest.raises(ValueError, match=rf"data\.txt:3: .*{msg}"):
        sl.parse_trajectories(path)


def _golden_file(tmp_path, g):
    from oracle import sl_ref
    return sl_ref.write_lines(tmp_path / "golden.txt", sl_ref.golden_lines(g))


def test_deal_packing_matches_the_golden_boards(tmp_path):
    """The chance order of the golden lines (card at chance position k -> seat k mod 4 from North) packs back into the
    boards' hands."""
    from brl_b200 import sl
    g = _golden()
    t = sl.parse_trajectories(_golden_file(tmp_path, g))
    assert np.array_equal(t.table, g["table"])
    assert (t.table[:, 32:] == 0).all()                # no double-dummy results in the bidding data
    # the label of every golden example is the call stored at its position
    assert np.array_equal(t.calls[t.offsets[g["line"]] + g["position"]], g["label"])
    n_calls = np.diff(t.offsets)
    assert (n_calls == 4).sum() >= 10                  # passed-out deals (56-int lines) are in the fixture
    assert np.array_equal(np.bincount(g["line"], minlength=len(t)), n_calls)   # one example per call position


def test_oracle_replay_reproduces_the_reference_examples(tmp_path):
    """make_dataset's (observation, legal mask, label) for every (line, position) of the golden, bit for bit."""
    from brl_b200 import sl
    from oracle import sl_ref
    g = _golden()
    t = sl.parse_trajectories(_golden_file(tmp_path, g))
    obs, mask, label = sl_ref.replay_examples(t.table, t.calls, t.offsets, g["line"], g["position"])
    assert np.array_equal(np.packbits(obs, axis=1, bitorder="little"), g["obs_bits"])
    assert np.array_equal(mask, g["mask"])
    assert np.array_equal(label, g["label"])


def test_shuffled_stream_is_one_example_per_trajectory_per_pass():
    from brl_b200.sl import ShuffledStream
    s = ShuffledStream(10, seed=3)
    x = np.concatenate([s.take(7), s.take(7), s.take(6)])  # batches straddle the passes
    assert sorted(x[:10]) == list(range(10)) and sorted(x[10:]) == list(range(10))
    assert not np.array_equal(x[:10], x[10:])               # every pass is a fresh shuffle
    assert np.array_equal(ShuffledStream(10, seed=3).take(20), x)


def test_default_config_has_the_slconfig_fields():
    from brl_b200 import sl
    assert sl.default_config() == dict(iterations=400000, train_batch=128, learning_rate=1e-4, eval_every=10000,
                                       data_path=None, save_path=None, num_examples=3, eval_batch=10000, rng_seed=42,
                                       entropy_coef=0.0, type_of_model="DeepMind", activation="relu")


def test_sl_ref_target_loss_is_cross_entropy_over_38_entries():
    """-mean(one_hot * log_softmax) averages over B * 38 entries: equal logits give log(38) / 38 per sample."""
    from oracle import sl_ref
    logits = torch.zeros((2, 38), dtype=torch.float64, requires_grad=True)
    labels = torch.tensor([0, 5])
    legal = torch.ones((2, 38), dtype=torch.bool)
    total, (target, entropy) = sl_ref.loss(logits, labels, legal)
    target = target.detach()
    assert float(target) == pytest.approx(np.log(38) / 38, rel=1e-12)
    assert float(total.detach()) == float(target)
    total.backward()
    # d/dl_j = (1/38 - [j == label]) / (38 * B)
    want = (np.full((2, 38), 1 / 38) - np.eye(38)[[0, 5]]) / (38 * 2)
    np.testing.assert_allclose(logits.grad.numpy(), want, rtol=1e-12, atol=1e-15)


def test_sl_ref_entropy_is_over_the_legal_calls_only():
    from oracle import sl_ref
    logits = torch.zeros((1, 38), dtype=torch.float64)
    logits[0, 7] = 100.0                                 # large but illegal: ignored by the entropy, not by the target
    legal = torch.zeros((1, 38), dtype=torch.bool)
    legal[0, [0, 1, 3, 4]] = True
    total, (target, entropy) = sl_ref.loss(logits, torch.tensor([0]), legal, entropy_coef=0.5)
    assert float(entropy) == pytest.approx(np.log(4), rel=1e-12)
    assert float(target) == pytest.approx(100.0 / 38, rel=1e-6)        # -log softmax(l)[0] ~ 100, over 38 entries
    assert float(total) == pytest.approx(float(target) - 0.5 * np.log(4), rel=1e-12)
    m = sl_ref.test_metrics(logits, torch.tensor([7]), legal)
    assert m["test/test_accuracy"] == 1.0 and m["test/illegal_actions_prob"] == pytest.approx(1.0, abs=1e-12)


def test_sl_ref_adam_two_steps_eps_1e8_no_clipping():
    """optax.adam(lr): the bias-corrected first step is lr * sign(g) (up to eps); no clipping however large g is."""
    from oracle import sl_ref
    p, m, v = np.zeros(3), np.zeros(3), np.zeros(3)
    g1 = np.array([1e6, -2.0, 0.0])
    p, m, v = sl_ref.adam_step(p, g1, m, v, 0, lr=0.1)
    np.testing.assert_allclose(p, [-0.1, 0.1, 0.0], rtol=1e-8)   # eps / |g| of the step
    g2 = np.array([1e6, 2.0, 1e-9])
    p1 = p.copy()
    p, m, v = sl_ref.adam_step(p, g2, m, v, 1, lr=0.1)
    m_hat = (0.9 * 0.1 * g1 + 0.1 * g2) / (1 - 0.9 ** 2)
    v_hat = (0.999 * 0.001 * g1 ** 2 + 0.001 * g2 ** 2) / (1 - 0.999 ** 2)
    want = p1 - 0.1 * m_hat / (np.sqrt(v_hat) + 1e-8)
    np.testing.assert_allclose(p, want, rtol=1e-12)
    assert p[0] == pytest.approx(-0.2, rel=1e-9)        # no clip_by_global_norm: the 1e6 gradient takes a full step
    # eps = 1e-8, not ppo's 1e-5: a 1e-9 gradient still moves its parameter by a visible fraction of lr
    assert abs(p[2]) > 0.01 * 0.1


def test_train_refuses_the_nets_the_hot_path_does_not_run():
    from brl_b200 import sl
    for cfg in ({"type_of_model": "FAIR"}, {"activation": "tanh"}):
        with pytest.raises(NotImplementedError):
            sl.train(cfg, train="unused", test="unused", device="cpu")
