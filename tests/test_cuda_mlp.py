"""GPU parity of the tcgen05 policy forward (csrc/brl_mlp.cu) against the oracle's NumPy
restatement of src/models.py:23-33, on real observations produced by the env kernels.

Tolerances (floating point, stated here as the north star asks): the reference computes in
fp32; the default "tc" mode (3-term bf16 split, fp32 accumulation in TMEM) must agree with a
float64 evaluation to 5e-5 of the output range -- the same order as fp32 GEMM round-off -- and
pick the same argmax wherever the float64 top-2 gap exceeds 1e-4; the single-product
"tc-bf16" mode is held to 2e-2 (it is an opt-in speed mode, not the parity path)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FORCE_LAYERS = 1 << 29  # BRL_F_TUNE_MLP_LAYERS (include/brl_b200.h)


def _real_obs(n, steps=9, seed=11):
    from brl_b200 import ops
    from brl_b200.deals import synthetic_deal_table
    table = torch.as_tensor(synthetic_deal_table(500, 2), device=DEV)
    state, out = ops.new_state(n, DEV), ops.EnvOutputs(n, DEV)
    ops.init(ops.make_keys(seed, n, DEV), table, state, out)
    for i in range(steps):
        ops.step(state, None, table, state, out, autoreset=True, random_action=True, seed=seed, step_index=i)
    return out.observation


def _params(seed):
    from brl_b200.models import LAYERS, init_params
    params = init_params(seed, DEV)
    g = torch.Generator(device="cpu").manual_seed(seed)
    for name in LAYERS:  # non-zero biases so the bias path is exercised
        params[name]["b"] = (torch.randn(params[name]["b"].shape, generator=g) * 0.1).to(DEV)
    return params


def _ref64(params, x):
    from brl_b200.models import params_to_numpy
    from oracle import oracle as orc
    flat = {k: v.astype(np.float64) for k, v in params_to_numpy(params).items()}
    return orc.mlp_forward(flat, x.cpu().numpy().astype(np.float64))


@pytest.mark.parametrize("n", [1, 100, 128, 1000, 8192 + 77])
def test_tc_forward_matches_float64_reference(n):
    from brl_b200.models import make_forward_pass
    params = _params(n)
    x = _real_obs(n)
    l64, v64 = _ref64(params, x)
    logits, value = make_forward_pass(precision="tc").apply(params, x)
    logits, value = logits.cpu().numpy(), value.cpu().numpy()
    assert logits.shape == (n, 38) and value.shape == (n,)
    scale_l, scale_v = np.abs(l64).max(), max(np.abs(v64).max(), 1e-3)
    assert np.abs(logits - l64).max() <= 5e-5 * scale_l
    assert np.abs(value - v64).max() <= 5e-5 * scale_v
    top2 = np.sort(l64, axis=1)[:, -2:]
    decided = (top2[:, 1] - top2[:, 0]) > 1e-4
    assert (logits.argmax(1)[decided] == l64.argmax(1)[decided]).all()


def test_tc_forward_tracks_cublas_fp32():
    """independent cross-check against the library GEMM chain (cuBLAS fp32 through torch)"""
    from brl_b200.models import make_forward_pass
    from scripts.torch_baseline import TorchForwardPass
    params = _params(3)
    x = _real_obs(4096)
    lt, vt = make_forward_pass(precision="tc").apply(params, x)
    lf, vf = TorchForwardPass("relu", "fp32").apply(params, x)
    assert float((lt - lf).abs().max()) <= 5e-5 * float(lf.abs().max())
    assert float((vt - vf).abs().max()) <= 5e-5 * max(float(vf.abs().max()), 1e-3)


def test_tc_bf16_mode_and_input_dtypes():
    from brl_b200 import ops
    from brl_b200.models import make_forward_pass
    params = _params(4)
    x = _real_obs(777)
    l64, v64 = _ref64(params, x)
    lb, vb = make_forward_pass(precision="tc-bf16").apply(params, x)
    assert np.abs(lb.cpu().numpy() - l64).max() <= 2e-2 * np.abs(l64).max()
    # u8 / bool / bf16 observations feed the same kernels and give identical results
    fp = make_forward_pass(precision="tc")
    base, _ = fp.apply(params, x)
    for xx in (x.to(torch.uint8), x.to(torch.bool), ops.obs_to_bf16(x)):
        l2, _ = fp.apply(params, xx)
        assert torch.equal(l2, base)


def test_repack_after_in_place_update():
    from brl_b200.models import LAYERS, make_forward_pass
    params = _params(5)
    x = _real_obs(256)
    fp = make_forward_pass(precision="tc")
    l0, _ = fp.apply(params, x)
    params[LAYERS[4]]["b"].add_(1.0)  # optimizer-style in-place update
    l1, _ = fp.apply(params, x)
    assert torch.allclose(l1, l0 + 1.0, atol=1e-5)


@pytest.mark.parametrize("n", [100, 4096 + 33, 8192])
@pytest.mark.parametrize("sample", [False, True])
def test_policy_act_equals_forward_then_categorical(n, sample):
    """brl_policy_act (one persistent launch from 4096 envs on: the head-tile epilogue samples in place) against
    brl_mlp_forward + brl_categorical: identical logits / value bits and identical actions (same Philox noise, same
    tie rule); log_prob within 2e-6 absolute (the fused row sums exp() sequentially, the warp kernel as a tree)."""
    from brl_b200 import ops
    from brl_b200.deals import synthetic_deal_table
    params = _params(3)
    from brl_b200.models import LAYERS
    blob = ops.mlp_pack([params[k]["w"] for k in LAYERS], [params[k]["b"] for k in LAYERS])
    table = torch.as_tensor(synthetic_deal_table(500, 2), device=DEV)
    state, out = ops.new_state(n, DEV), ops.EnvOutputs(n, DEV, torch.bfloat16)
    ops.init(ops.make_keys(5, n, DEV), table, state, out)
    for i in range(6):
        ops.step(state, None, table, state, out, autoreset=True, random_action=True, seed=5, step_index=i)
    x, mask = out.observation, out.legal_action_mask
    scratch = ops.mlp_scratch(n, DEV)
    lg, vl = torch.empty((n, 38), device=DEV), torch.empty(n, device=DEV)
    ops.mlp_forward(x, blob, scratch, lg, vl)
    a_ref, lp_ref = torch.empty(n, dtype=torch.int32, device=DEV), torch.empty(n, device=DEV)
    for use_mask in (True, False):
        m = mask if use_mask else None
        ops.categorical(lg, m, a_ref, lp_ref, sample=sample, seed=99, env_offset=1000)
        a, lp, v2, lg2 = torch.full_like(a_ref, -7), torch.full_like(lp_ref, float("nan")), torch.empty_like(vl), torch.empty_like(lg)
        ops.policy_act(x, blob, scratch, m, a, lp, v2, lg2, sample=sample, seed=99, env_offset=1000)
        assert torch.equal(lg2, lg) and torch.equal(v2, vl)
        assert torch.equal(a, a_ref)
        assert float((lp - lp_ref).abs().max()) <= 2e-6
        if use_mask:
            assert bool(mask.gather(1, a.long()[:, None]).all()), "sampled an illegal action"
        # optional outputs may be omitted
        a3 = torch.full_like(a_ref, -7)
        ops.policy_act(x, blob, scratch, m, a3, sample=sample, seed=99, env_offset=1000)
        assert torch.equal(a3, a_ref)


@pytest.mark.parametrize("n,tune", [(100, 0), (4096, FORCE_LAYERS)])
def test_seed_salt_is_refused_off_the_fused_launch(n, tune):
    """BRL_F_SEED_SALT is read by the fused launch only: a salted call that runs on the per-layer launches, by its size or
    forced there, is an error (BRL_E_OPAQUE) rather than a sample drawn with the unsalted seed"""
    from brl_b200 import _lib, ops
    obs = torch.zeros((n, 480), dtype=torch.bfloat16, device=DEV)
    blob = torch.zeros(_lib.load().brl_mlp_packed_bytes(), dtype=torch.uint8, device=DEV)
    action = torch.full((n,), -7, dtype=torch.int32, device=DEV)
    salt = torch.zeros(1, dtype=torch.int64, device=DEV)
    with pytest.raises(_lib.BrlError, match=r"\(-1\).*SEED_SALT"):
        ops.policy_act(obs, blob, ops.mlp_scratch(n, DEV), None, action, sample=True, tune=tune, seed_salt=salt)
    assert bool((action == -7).all())


def test_product_forward_has_no_library_back_end():
    """north_star: no multi-backend dispatch.  The product's forward pass is the tensor-core kernel or nothing."""
    from brl_b200.models import make_forward_pass
    for bad in ("fp32", "tf32", "bf16"):
        with pytest.raises(ValueError):
            make_forward_pass(precision=bad)
    with pytest.raises(NotImplementedError):
        make_forward_pass(activation="tanh")
    with pytest.raises(NotImplementedError):
        make_forward_pass(model_type="FAIR")


def test_team_rows_lists_live_envs_by_acting_team():
    from brl_b200 import ops
    for n in (1, 37, 1024, 5000, 70_001):
        g = torch.Generator(device=DEV).manual_seed(n)
        player = torch.randint(0, 4, (n,), generator=g, device=DEV).to(torch.int8)
        done = (torch.rand(n, generator=g, device=DEV) < 0.4).to(torch.uint8)
        r1, r2 = torch.full((n,), -1, dtype=torch.int32, device=DEV), torch.full((n,), -1, dtype=torch.int32, device=DEV)
        counts = torch.full((2,), 99, dtype=torch.int32, device=DEV)
        ops.team_rows(player, done, r1, r2, counts)
        c1, c2 = counts.tolist()
        want1 = torch.nonzero((done == 0) & (player < 2))[:, 0].to(torch.int32)
        want2 = torch.nonzero((done == 0) & (player >= 2))[:, 0].to(torch.int32)
        assert c1 == want1.numel() and c2 == want2.numel()
        assert torch.equal(torch.sort(r1[:c1]).values, want1) and torch.equal(torch.sort(r2[:c2]).values, want2)
        # rows ascend inside each 1024-env block (ballot order)
        if n <= 1024:
            assert torch.equal(r1[:c1], want1) and torch.equal(r2[:c2], want2)
        ops.team_rows(player, None, r1, r2, counts)   # done = NULL: every env is live
        assert int(counts.sum()) == n


@pytest.mark.parametrize("n,n_rows", [(300, 100), (9000, 4096 + 77), (20_000, 13_000)])
@pytest.mark.parametrize("sample", [False, True])
def test_policy_act_rows_equals_full_policy_act_on_the_listed_envs(n, n_rows, sample):
    """the listed forward (gather -> net -> scatter by env) gives bit-identical action / log_prob / logits to the full-batch
    call for the listed envs and leaves every other entry untouched -- below and above the fused-launch size"""
    from brl_b200 import ops
    from brl_b200.models import make_forward_pass
    params = _params(6)
    x = ops.obs_to_bf16(_real_obs(n))
    g = torch.Generator(device=DEV).manual_seed(5)
    mask = (torch.rand((n, 38), generator=g, device=DEV) < 0.5).to(torch.uint8)
    mask[:, 0] = 1
    fp = make_forward_pass(precision="tc")
    packed = fp._packed(params)
    a_full = torch.empty(n, dtype=torch.int32, device=DEV)
    lp_full = torch.empty(n, dtype=torch.float32, device=DEV)
    lg_full = torch.empty((n, 38), dtype=torch.float32, device=DEV)
    ops.policy_act(x, packed, ops.mlp_scratch(n, DEV), mask, a_full, lp_full, None, lg_full, sample=sample, seed=77, env_offset=1000)
    rows = torch.randperm(n, generator=g, device=DEV)[:n_rows].to(torch.int32).contiguous()
    a = torch.full((n,), -5, dtype=torch.int32, device=DEV)
    lp = torch.full((n,), 9.0, dtype=torch.float32, device=DEV)
    lg = torch.full((n, 38), 7.0, dtype=torch.float32, device=DEV)
    ops.policy_act_rows(x, packed, ops.mlp_rows_scratch(n_rows, DEV), mask, a, rows, lp, lg, sample=sample, seed=77, env_offset=1000)
    sel = torch.zeros(n, dtype=torch.bool, device=DEV)
    sel[rows.long()] = True
    assert torch.equal(a[sel], a_full[sel]) and torch.equal(lp[sel], lp_full[sel]) and torch.equal(lg[sel], lg_full[sel])
    assert bool((a[~sel] == -5).all()) and bool((lp[~sel] == 9.0).all()) and bool((lg[~sel] == 7.0).all())
