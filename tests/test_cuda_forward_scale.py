"""Float64 parity of the tensor-core policy forward (csrc/brl_mlp.cu) and of the PPO update GEMMs (csrc/brl_mlp_train.cu) at
league scale, on both launch paths, with the caller's scratch poisoned before every checked call.

The other forward tests compare the kernel with float64 up to 8,269 rows (about one wave of the fused launch) and above that
with other calls of the same kernel.  Here every output is compared with an independent float64 evaluation of the net
(`ref_forward`: torch GEMMs in float64 on the device, nothing shared with the kernel) from one row to 262,477 rows (about
17,400 tiles over the CTA pairs), on the fused launch forced down to one row and the per-layer launches forced up to 65,536
rows.

Bar (DESIGN section 5): logits and value within 5e-5 of the output range, the range taken per 256-row block (the fused tile
height), so a block of extreme rows cannot hide a small-magnitude block next to it; decisions equal to the float64 masked
argmax wherever the float64 top-2 gap exceeds 1e-4 of the block's range; log_prob within the bar of the float64 masked
log-softmax.  The single-product "tc-bf16" mode keeps its 2e-2 bar.

Scratch is filled with 0xFF bytes before every checked call: NaN as bf16 activations and 0xFFFFFFFF as the fused launch's
tile counters, so a tile that read a layer's rows before they were published, or a counter the launch did not zero, shows
up as a NaN or a wrong row instead of the plausible values an earlier call left behind.  Outputs start as NaN / -7 and must
all be written.

The CPU part shows that the bar can fail: an emulation of the kernel's split-bf16 arithmetic passes it, a single bf16 product
does not, and each of a set of plausible kernel bugs applied to the reference fails it."""
import numpy as np
import pytest
import torch

from tests import helpers as H

DEV = "cuda:0"
FORCE_LAYERS = 1 << 29  # BRL_F_TUNE_MLP_LAYERS (include/brl_b200.h)
FORCE_FUSED = 1 << 30   # BRL_F_TUNE_MLP_FUSED
BLOCK = 256             # rows of one fused tile (a CTA pair's row block); the bar's range is taken per block
BAR, BAR_BF16, GAP = 5e-5, 2e-2, 1e-4
CHUNK = 32768           # rows per float64 reference GEMM chain
TAG_GUM = 0x47554D30    # Philox counter tag of the Gumbel noise (brl_categorical, oracle/brl_oracle.c)


# ---- float64 reference and bar -------------------------------------------------------------------------------------------
def ref_forward(params, x, device, hook=None):
    """The DeepMind MLP (src/models.py:23-33) in float64 torch on `device`, in row chunks of at most CHUNK rows.
    `hook(layer, row0, h)` may return a replacement for hidden layer `layer`'s input (rows row0.. of the batch): it is how
    the mutation checks plant a kernel bug.  -> (logits f64[n, 38], value f64[n]) on `device`."""
    from brl_b200.models import LAYERS
    w = [params[k]["w"].to(device=device, dtype=torch.float64) for k in LAYERS]
    b = [params[k]["b"].to(device=device, dtype=torch.float64) for k in LAYERS]
    head_w, head_b = torch.cat([w[4], w[5]], 1), torch.cat([b[4], b[5]])
    out = []
    for r0 in range(0, x.shape[0], CHUNK):
        h = x[r0:r0 + CHUNK].to(device=device, dtype=torch.float64)
        for i in range(4):
            if hook is not None:
                h = hook(i, r0, h)
            h = torch.relu(h @ w[i] + b[i])
        out.append(h @ head_w + head_b)
    z = torch.cat(out)
    return z[:, :38].contiguous(), z[:, 38].contiguous()


def block_range(want, floor=1e-3):
    """per row: the largest |want| over the row's 256-row block (at least `floor`, so all-zero outputs keep a bar).  The
    last block of a ragged batch is ranged over the batch's last 256 rows: a tail of a few rows has no output range of its
    own (one row's value is a single number, often a small difference of large terms)"""
    n = want.shape[0]
    m = want.reshape(n, -1).abs().amax(1)
    full = n // BLOCK
    out = torch.empty_like(m)
    if full:
        out[:full * BLOCK] = m[:full * BLOCK].view(full, BLOCK).amax(1).repeat_interleave(BLOCK)
    if n > full * BLOCK:
        out[full * BLOCK:] = m[max(0, n - BLOCK):].amax()
    return out.clamp_min(floor)


def err_ratio(got, want, bar=BAR):
    """per row: max |got - want| over the row / (bar * its block's range); > 1 fails"""
    n = want.shape[0]
    err = (got.to(want.dtype) - want).abs().reshape(n, -1).amax(1)
    return err / (bar * block_range(want))


def masked_top2(logits, mask):
    """float64 masked argmax and the gap to the runner-up (inf where a single action is legal)"""
    ml = logits if mask is None else logits.masked_fill(mask == 0, float("-inf"))
    top = ml.topk(2, dim=1)
    gap = top.values[:, 0] - top.values[:, 1]
    return top.indices[:, 0], torch.nan_to_num(gap, nan=float("inf"), posinf=float("inf"))


def _worst(ratio, what):
    r, i = (float(v) for v in ratio.max(0))
    assert r <= 1.0, f"{what} {r:.3g} x the bar at row {int(i)}"
    return r


def check_forward(lg, vl, l64, v64, bar=BAR, what=""):
    """every output written and finite, logits and value within the bar; -> worst error / bar of (logits, value)"""
    assert bool(torch.isfinite(lg).all()) and bool(torch.isfinite(vl).all()), f"{what}: an output was not written"
    return _worst(err_ratio(lg, l64, bar), f"{what}: logits"), _worst(err_ratio(vl, v64, bar), f"{what}: value")


def check_decisions(action, l64, mask, what=""):
    """the masked argmax equals float64's wherever the float64 top-2 gap exceeds GAP of the block's range"""
    a64, gap = masked_top2(l64, mask)
    decided = gap > GAP * block_range(l64)
    bad = decided & (action.long() != a64)
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} decisions differ from float64 (first row {int(bad.nonzero()[0])})"


def check_log_prob(log_prob, action, l64, mask, what=""):
    """log_prob of the chosen action within the bar of the float64 masked log-softmax; -> worst error / bar"""
    assert bool(torch.isfinite(log_prob).all()), f"{what}: log_prob not written"
    ml = l64 if mask is None else l64.masked_fill(mask == 0, float("-inf"))
    lp64 = torch.log_softmax(ml, 1).gather(1, action.long()[:, None])[:, 0]
    return _worst((log_prob.double() - lp64).abs() / (BAR * block_range(l64)), f"{what}: log_prob")


# ---- nets and inputs ------------------------------------------------------------------------------------------------------
def biased_params(seed, device):
    """haiku init (models.init_params) with non-zero biases, so that every bias path is exercised"""
    from brl_b200.models import LAYERS, init_params
    p = init_params(seed, device)
    g = torch.Generator().manual_seed(seed)
    for name in LAYERS:
        p[name]["b"] = (torch.randn(p[name]["b"].shape, generator=g) * 0.1).to(device)
    return p


def wide_params(seed, device):
    """hidden columns scaled by 2^u, u uniform in [-6, 6]: every row of the next layer's input mixes magnitudes 2^12 apart,
    where the split's hi / lo terms and the fp32 accumulation matter"""
    from brl_b200.models import LAYERS
    p = biased_params(seed, device)
    g = torch.Generator().manual_seed(seed + 1)
    for name in LAYERS[:4]:
        s = torch.exp2(torch.rand(p[name]["b"].shape, generator=g) * 12 - 6).to(device)
        p[name]["w"] *= s
        p[name]["b"] *= s
    return p


NETS = {"biased": biased_params, "seeded": H.seeded_params, "wide": wide_params}


def random_bits(n, density, seed, device):
    g = torch.Generator(device=device).manual_seed(seed)
    return (torch.rand((n, 480), generator=g, device=device) < density).to(torch.bfloat16)


# ---- emulation of the kernel's arithmetic (CPU) ------------------------------------------------------------------------------
def _bf16(t):
    return t.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def emulate_forward(params, x, single_bf16):
    """the kernel's arithmetic in float64: weights and activations as bf16 hi (+ lo = bf16(v - hi)); the split mode sums
    x_hi w_hi + x_lo w_hi + x_hi w_lo (the 0/1 observation is exact: two terms), the single mode x_hi w_hi; every layer's
    output rounded to fp32"""
    from brl_b200.models import LAYERS
    w = [params[k]["w"].double().cpu() for k in LAYERS]
    b = [params[k]["b"].double().cpu() for k in LAYERS]
    ws, bs = w[:4] + [torch.cat([w[4], w[5]], 1)], b[:4] + [torch.cat([b[4], b[5]])]
    h = x.double().cpu()
    for i in range(5):
        w_hi = _bf16(ws[i])
        w_lo = _bf16(ws[i] - w_hi)
        h_hi = _bf16(h)
        if single_bf16:
            z = h_hi @ w_hi
        else:
            h_lo = _bf16(h - h_hi)
            z = h_hi @ w_hi + h_lo @ w_hi + h_hi @ w_lo
        z = (z + bs[i]).float().double()
        h = torch.relu(z) if i < 4 else z
    return h[:, :38].contiguous(), h[:, 38].contiguous()


def _emulation_case(density, seed=3, n=1024):
    p = biased_params(seed, "cpu")
    p["actor_critic/linear_4"]["w"] *= 128  # a trained net's logit magnitude (helpers.seeded_params)
    return p, (torch.rand((n, 480), generator=torch.Generator().manual_seed(seed)) < density).float()


def test_reference_matches_the_oracle():
    """ref_forward (torch float64) against oracle.mlp_forward (NumPy) on a few hundred rows, two nets"""
    from brl_b200.models import params_to_numpy
    from oracle import oracle as orc
    for make in (biased_params, wide_params):
        p = make(7, "cpu")
        x = (torch.rand((300, 480), generator=torch.Generator().manual_seed(1)) < 0.2).float()
        l64, v64 = ref_forward(p, x, "cpu")
        flat = {k: v.astype(np.float64) for k, v in params_to_numpy(p).items()}
        lo, vo = orc.mlp_forward(flat, x.numpy())
        assert np.abs(l64.numpy() - lo).max() <= 1e-12 * np.abs(lo).max()
        assert np.abs(v64.numpy() - vo).max() <= 1e-12 * max(np.abs(vo).max(), 1e-3)


@pytest.mark.parametrize("density", [0.05, 0.3])
def test_bar_passes_the_split_and_fails_a_single_bf16_product(density):
    """the bar sits between the two arithmetics: the split emulation passes it (measured ~0.2 of the bar), the single bf16
    product fails it on most row blocks (~100 x the bar)"""
    p, x = _emulation_case(density)
    l64, v64 = ref_forward(p, x, "cpu")
    ls, vs = emulate_forward(p, x, single_bf16=False)
    assert float(err_ratio(ls, l64).max()) <= 0.5 and float(err_ratio(vs, v64).max()) <= 0.5
    lb, _ = emulate_forward(p, x, single_bf16=True)
    failed = (err_ratio(lb, l64).view(-1, BLOCK).amax(1) > 1.0).float().mean()
    assert float(failed) > 0.5
    # the single product stays inside the 2e-2 bar of the tc-bf16 mode
    assert float(err_ratio(lb, l64, BAR_BF16).max()) <= 0.5


def test_wide_net_emulation_passes_the_bar():
    """the wide-range net's hidden columns span 2^12: the split arithmetic still passes the bar, the single product its own"""
    p = wide_params(5, "cpu")
    x = (torch.rand((512, 480), generator=torch.Generator().manual_seed(2)) < 0.3).float()
    l64, v64 = ref_forward(p, x, "cpu")
    ls, vs = emulate_forward(p, x, single_bf16=False)
    assert float(err_ratio(ls, l64).max()) <= 0.5 and float(err_ratio(vs, v64).max()) <= 0.5
    lb, _ = emulate_forward(p, x, single_bf16=True)
    assert float(err_ratio(lb, l64, BAR_BF16).max()) <= 0.5


def _swap_chunks(layer, r0, h):  # two 16-byte (8-column) chunks of layer 0's input swapped inside one 128-byte swizzle row
    if layer == 0:
        h = h.clone()
        h[:, 8:16], h[:, 16:24] = h[:, 16:24].clone(), h[:, 8:16].clone()
    return h


def _drop_last_k_block(layer, r0, h):  # layer 0's last K block (columns 448-479, the hand) never loaded
    if layer == 0:
        h = h.clone()
        h[:, 448:] = 0
    return h


def _rank1_reads_rank0(layer, r0, h):  # the rank-1 half of row block 1 reads layer 2's input from the rank-0 half's rows
    if layer == 2:
        h = h.clone()
        h[BLOCK + 128:2 * BLOCK] = h[BLOCK:BLOCK + 128]
    return h


@pytest.mark.parametrize("bug", [_swap_chunks, _drop_last_k_block, _rank1_reads_rank0], ids=lambda f: f.__name__.strip("_"))
@pytest.mark.parametrize("density", [0.05, 0.3])
def test_planted_kernel_bugs_fail_the_bar(bug, density):
    p, x = _emulation_case(density, n=512)
    l64, v64 = ref_forward(p, x, "cpu")
    lm, vm = ref_forward(p, x, "cpu", hook=bug)
    ratio = torch.maximum(err_ratio(lm, l64), err_ratio(vm, v64))
    assert float(ratio.max()) > 10.0
    if bug is _rank1_reads_rank0:  # only the planted rows are off
        assert float(ratio[:BLOCK + 128].max()) == 0.0 and float(ratio[BLOCK + 128:].min()) > 1.0


def test_neighbouring_pool_net_bias_fails_the_bar():
    """grouped forward: row block 1 runs net 1's weights but one layer's bias of net 0, the pool's neighbour"""
    from brl_b200.models import LAYERS
    nets = [biased_params(11, "cpu"), biased_params(12, "cpu")]
    x = (torch.rand((2 * BLOCK, 480), generator=torch.Generator().manual_seed(4)) < 0.05).float()
    want = [ref_forward(nets[m], x[m * BLOCK:(m + 1) * BLOCK], "cpu") for m in range(2)]
    l64, v64 = torch.cat([w[0] for w in want]), torch.cat([w[1] for w in want])
    for layer in range(5):
        bad = {k: dict(v) for k, v in nets[1].items()}
        bad[LAYERS[layer]]["b"] = nets[0][LAYERS[layer]]["b"]
        lb, vb = ref_forward(bad, x[BLOCK:], "cpu")
        ratio = torch.maximum(err_ratio(torch.cat([want[0][0], lb]), l64), err_ratio(torch.cat([want[0][1], vb]), v64))
        assert float(ratio.max()) > 10.0, layer


# ---- forward at scale, both paths, poisoned scratch (GPU) ----------------------------------------------------------------------
SIZES = [1, 127, 128, 129, 255, 256, 257, 4095, 4096, 4097, 8192 + 77, 65_536, 262_144 + 333]
CASES = [(n, 0) for n in SIZES] + [(n, FORCE_FUSED) for n in (1, 129, 257, 4095)] + [(n, FORCE_LAYERS) for n in (4097, 65_536)]
_TABLE = {}


def _path(n, tune):
    return "fused" if tune == FORCE_FUSED or (tune == 0 and n >= 4096) else "layers"


def _case_id(case):
    n, tune = case
    return f"{n}-{'default' if tune == 0 else _path(n, tune)}"


def _env_obs(n, steps, seed):
    """observations (bf16) and legal masks of n envs after `steps` random-legal auto-reset steps"""
    from brl_b200 import ops
    from brl_b200.deals import synthetic_deal_table
    if "t" not in _TABLE:
        _TABLE["t"] = torch.as_tensor(synthetic_deal_table(500, 2), device=DEV)
    table = _TABLE["t"]
    state, out = ops.new_state(n, DEV), ops.EnvOutputs(n, DEV, torch.bfloat16)
    ops.init(ops.make_keys(seed, n, DEV), table, state, out)
    for i in range(steps):
        ops.step(state, None, table, state, out, autoreset=True, random_action=True, seed=seed, step_index=i)
    return out.observation, out.legal_action_mask


def make_inputs(n, seed):
    """n rows, shuffled: a quarter each of env observations after 9 and after 30 random steps (late-auction X / XX columns)
    with their legal masks, and of random bits at densities 0.05 and 0.5 with random masks; all-zero rows at 127, 255 and
    the second-to-last row, all-one rows at 128, 256 and the last row (tile boundaries of both paths)"""
    q = n // 4
    parts, masks = [], []
    g = torch.Generator(device=DEV).manual_seed(seed)
    for kind, k in (("env9", n - 3 * q), ("env30", q), ("bits0.05", q), ("bits0.5", q)):
        if k == 0:
            continue
        if kind.startswith("env"):
            o, m = _env_obs(k, int(kind[3:]), seed + k)
        else:
            o = random_bits(k, float(kind[4:]), seed + k, DEV)
            m = (torch.rand((k, 38), generator=g, device=DEV) < 0.5).to(torch.uint8)
            m[:, 0] = 1
        parts.append(o)
        masks.append(m)
    perm = torch.randperm(n, generator=g, device=DEV)
    x, mask = torch.cat(parts)[perm].contiguous(), torch.cat(masks)[perm].contiguous()
    for r in (127, 255, n - 2):
        if 0 <= r < n:
            x[r] = 0
    for r in (128, 256, n - 1):
        if 0 <= r < n:
            x[r] = 1
    return x, mask


def _nan(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device=DEV)


def check_sample(action, l64, mask, seed, env_offset, step, what=""):
    """Gumbel-argmax samples against oracle.categorical on the float64 logits: the same action except where the two
    Gumbel-perturbed float64 values are within the bar of each other (the noise is recomputed from the oracle's Philox)"""
    from oracle import oracle as orc
    n = l64.shape[0]
    assert bool(mask.gather(1, action.long()[:, None]).all()), f"{what}: sampled an illegal action"
    a_k = action.cpu().numpy()
    a_o, _ = orc.categorical(l64.float().cpu().numpy(), mask.cpu().numpy(), True, seed, env_offset, step)
    diff = np.nonzero(a_k != a_o)[0]
    assert len(diff) <= 10 + n // 1000, f"{what}: {len(diff)} of {n} samples differ from the oracle's"
    if len(diff) == 0:
        return
    lg, rng = l64[diff].cpu().numpy(), block_range(l64)[diff].cpu().numpy()

    def perturbed(i, r, a):
        e = env_offset + int(r)
        w = orc.philox([e & 0xFFFFFFFF, e >> 32, TAG_GUM + a // 4, step], [seed & 0xFFFFFFFF, seed >> 32])[a % 4]
        u = (np.float32(w >> 8) + np.float32(0.5)) * np.float32(1.0 / 16777216.0)
        return lg[i, a] - np.log(-np.log(np.float64(u)))

    for i, r in enumerate(diff):
        gap = abs(perturbed(i, r, int(a_o[r])) - perturbed(i, r, int(a_k[r])))
        assert gap <= BAR * rng[i], f"{what}: row {r} sampled {a_k[r]}, the oracle {a_o[r]}, perturbed gap {gap:.3g}"


@pytest.mark.gpu
@pytest.mark.parametrize("n,tune", CASES, ids=[_case_id(c) for c in CASES])
def test_forward_matches_float64_at_scale(n, tune, record_property):
    """mlp_forward (tc, tc-bf16), policy_act (mode, sample) and policy_act_rows against float64 on three nets, scratch
    poisoned before every call; then two forwards with different nets and inputs back to back on one scratch"""
    from brl_b200 import ops
    from brl_b200.models import LAYERS
    x, mask = make_inputs(n, seed=n + tune % 97)
    scratch = ops.mlp_scratch(n, DEV)
    n_rows = max(1, n // 2)
    rows_scratch = ops.mlp_rows_scratch(n_rows, DEV)
    path = _path(n, tune)
    worst = {}

    def note(key, r):
        if isinstance(r, tuple):  # check_forward: (logits, value)
            note(key + " logits", r[0])
            note(key + " value", r[1])
        else:
            worst[key] = max(worst.get(key, 0.0), r)

    blobs, refs = {}, {}
    for k, (name, make) in enumerate(NETS.items()):
        params = make(1000 + n + k, DEV)
        blobs[name] = ops.mlp_pack([params[m]["w"] for m in LAYERS], [params[m]["b"] for m in LAYERS])
        l64, v64 = refs[name] = ref_forward(params, x, DEV)
        blob, what = blobs[name], f"n={n} {path} {name}"
        for single in (False, True):
            scratch.fill_(0xFF)
            lg, vl = _nan(n, 38), _nan(n)
            ops.mlp_forward(x, blob, scratch, lg, vl, single_bf16=single, tune=tune)
            if single:  # the opt-in speed mode: logits only, at its own bar
                assert bool(torch.isfinite(lg).all()) and bool(torch.isfinite(vl).all())
                note("mlp_forward tc-bf16 logits", _worst(err_ratio(lg, l64, BAR_BF16), f"{what} tc-bf16: logits"))
            else:
                note("mlp_forward tc", check_forward(lg, vl, l64, v64, what=what + " mlp_forward"))
                check_decisions(lg.argmax(1), l64, None, what + " mlp_forward")
        for sample in (False, True):
            scratch.fill_(0xFF)
            a, lp, vl, lg = torch.full((n,), -7, dtype=torch.int32, device=DEV), _nan(n), _nan(n), _nan(n, 38)
            seed, env_offset, step = 77 + n, 1000, 3
            ops.policy_act(x, blob, scratch, mask, a, lp, vl, lg, sample=sample, seed=seed, env_offset=env_offset, step_index=step,
                           tune=tune)
            w = f"{what} policy_act {'sample' if sample else 'mode'}"
            note(f"policy_act {'sample' if sample else 'mode'}", check_forward(lg, vl, l64, v64, what=w))
            note(f"policy_act {'sample' if sample else 'mode'} log_prob", check_log_prob(lp, a, l64, mask, w))
            if sample:
                check_sample(a, l64, mask, seed, env_offset, step, w)
            else:
                assert bool(mask.gather(1, a.long()[:, None]).all()), f"{w}: an illegal action"
                check_decisions(a, l64, mask, w)
        # the listed forward on a random duplicate-free half of the envs in random order; the others stay untouched
        rows = torch.randperm(n, generator=torch.Generator(device=DEV).manual_seed(n + k), device=DEV)[:n_rows].to(torch.int32)
        rows_scratch.fill_(0xFF)
        a, lp, lg = torch.full((n,), -7, dtype=torch.int32, device=DEV), _nan(n), _nan(n, 38)
        ops.policy_act_rows(x, blob, rows_scratch, mask, a, rows, lp, lg, tune=tune)
        r = rows.long()
        listed = torch.zeros(n, dtype=torch.bool, device=DEV)
        listed[r] = True
        w = f"{what} policy_act_rows"
        assert bool((a[~listed] == -7).all()) and bool(lp[~listed].isnan().all()) and bool(lg[~listed].isnan().all()), \
            f"{w}: an unlisted env was written"
        assert bool(torch.isfinite(lg[r]).all()), f"{w}: a listed env was not written"
        # blocks of the compact (listed) batch the kernel ran
        note("policy_act_rows logits", _worst(err_ratio(lg[r], l64[r]), f"{w}: logits (listed row)"))
        note("policy_act_rows log_prob", check_log_prob(lp[r], a[r], l64[r], mask[r], w))
        check_decisions(a[r], l64[r], mask[r], w)
    # two calls with different nets and inputs on one scratch, no synchronisation in between
    perm = torch.randperm(n, generator=torch.Generator(device=DEV).manual_seed(7), device=DEV)
    xp = x[perm].contiguous()
    scratch.fill_(0xFF)
    out = [(_nan(n, 38), _nan(n)) for _ in range(2)]
    ops.mlp_forward(x, blobs["wide"], scratch, *out[0], tune=tune)
    ops.mlp_forward(xp, blobs["seeded"], scratch, *out[1], tune=tune)
    note("mlp_forward tc", check_forward(*out[0], *refs["wide"], what=f"n={n} {path} back-to-back, first call"))
    l64, v64 = refs["seeded"]
    note("mlp_forward tc", check_forward(*out[1], l64[perm], v64[perm], what=f"n={n} {path} back-to-back, second call"))
    for key, r in worst.items():
        record_property(f"{path} {key}", round(r, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("n,tune", [(257, FORCE_FUSED), (4097, 0)], ids=["257-fused", "4097-default"])
def test_input_dtypes_on_the_fused_path(n, tune):
    """f32, u8, bool and bf16 observations through obs_to_bf16 feed the fused launch the same bits"""
    from brl_b200 import ops
    from brl_b200.models import LAYERS
    x, _ = make_inputs(n, seed=5)
    params = H.seeded_params(9, DEV)
    blob = ops.mlp_pack([params[m]["w"] for m in LAYERS], [params[m]["b"] for m in LAYERS])
    l64, v64 = ref_forward(params, x, DEV)
    scratch = ops.mlp_scratch(n, DEV)
    for src in (x.float(), x.to(torch.uint8), x.bool(), x):
        xb = ops.obs_to_bf16(src.contiguous())
        assert torch.equal(xb, x), src.dtype
        scratch.fill_(0xFF)
        lg, vl = _nan(n, 38), _nan(n)
        ops.mlp_forward(xb, blob, scratch, lg, vl, tune=tune)
        check_forward(lg, vl, l64, v64, what=f"{src.dtype}")


GROUPINGS = [([255, 256, 257, 1, 120_001], 0), ([255, 256, 257, 1, 120_001], FORCE_LAYERS),
             ([1, 255, 256, 257, 0], 0), ([1, 255, 256, 257, 0], FORCE_FUSED)]


@pytest.mark.gpu
@pytest.mark.parametrize("sizes,tune", GROUPINGS, ids=["120k-default", "120k-layers", "small-default", "small-fused"])
def test_grouped_forward_matches_each_nets_float64(sizes, tune, record_property):
    """policy_act_grouped over a pool of five distinct nets: every env's logits against ITS net's float64 output, its
    action against the float64 masked argmax; group sizes around the 256-row blocks, one group above 100k rows"""
    from brl_b200 import ops
    from brl_b200.models import make_forward_pass
    M, n = len(sizes), sum(sizes)
    nets = [biased_params(21, DEV), H.seeded_params(22, DEV), wide_params(23, DEV), biased_params(24, DEV), H.seeded_params(25, DEV)]
    pool = ops.mlp_pack_pool(nets, make_forward_pass().pack_into)
    g = torch.Generator(device=DEV).manual_seed(n)
    net = torch.repeat_interleave(torch.arange(M, device=DEV), torch.tensor(sizes, device=DEV))
    net = net[torch.randperm(n, generator=g, device=DEV)].to(torch.int32)
    env_models = torch.stack([net, net], 1).contiguous()
    player = torch.randint(0, 4, (n,), generator=g, device=DEV).to(torch.int8)
    x, mask = make_inputs(n, seed=n + 1)
    cap = ops.model_rows_capacity(n, M)
    rows = torch.empty(cap, dtype=torch.int32, device=DEV)
    block_model = torch.empty(cap // BLOCK, dtype=torch.int32, device=DEV)
    counts, offsets = torch.empty(M, dtype=torch.int32, device=DEV), torch.empty(M + 1, dtype=torch.int32, device=DEV)
    ops.model_rows(player, None, env_models, rows, counts, offsets, block_model)
    assert counts.tolist() == sizes
    off = offsets.tolist()
    scratch = torch.empty(ops.policy_grouped_scratch_bytes(n, M), dtype=torch.uint8, device=DEV).fill_(0xFF)
    action, logits = torch.full((n,), -7, dtype=torch.int32, device=DEV), _nan(n, 38)
    ops.policy_act_grouped(x, pool, scratch, mask, action, rows[:off[M]], block_model, logits, n_rows=offsets[M:],
                           tune=tune)
    assert bool(torch.isfinite(logits).all()) and bool((action >= 0).all()), "an env was not written"
    worst = 0.0
    for m in range(M):
        if sizes[m] == 0:
            continue
        envs = rows[off[m]:off[m] + sizes[m]].long()  # the kernel's order: blocks of the bar = the kernel's row blocks
        l64, _ = ref_forward(nets[m], x[envs], DEV)
        worst = max(worst, _worst(err_ratio(logits[envs], l64), f"net {m}: logits (group row)"))
        check_decisions(action[envs], l64, mask[envs], f"net {m}")
    record_property(f"{'fused' if tune == FORCE_FUSED or (tune == 0 and off[M] >= 4096) else 'layers'} policy_act_grouped",
                    round(worst, 4))


# ---- the PPO update's GEMMs (GPU) ------------------------------------------------------------------------------------------------
def _ppo_setup(total, seed):
    """a trajectory of `total` rows, a net with non-zero biases, and the rows whose float64 hidden pre-activations all stay
    2e-5 away from zero: the gradient is discontinuous at a ReLU kink, where the split forward's ~1e-6 error may flip a mask
    bit (test_cuda_ppo.py::test_ppo_grad_matches_float64_autograd draws its minibatches the same way)"""
    from brl_b200.models import params_to_numpy
    g = torch.Generator(device=DEV).manual_seed(seed)
    d = dict(dtype=torch.float64, device=DEV)
    obs = torch.rand((total, 480), generator=g, device=DEV) < 0.05
    mask = torch.rand((total, 38), generator=g, device=DEV) < 0.5
    mask[:, 0] = True
    action = ((torch.rand((total, 38), generator=g, device=DEV) + 1) * mask).argmax(1).to(torch.int32)  # a legal action
    traj = dict(obs=obs, mask=mask, action=action, old_lp=-torch.rand(total, generator=g, **d) * 3,
                old_v=torch.randn(total, generator=g, **d) * 0.3, adv=torch.randn(total, generator=g, **d),
                tgt=torch.randn(total, generator=g, **d) * 0.3)
    params = biased_params(seed, DEV)
    pn = {k: torch.tensor(v, **d) for k, v in params_to_numpy(params).items()}
    h, margin = obs.double(), torch.full((total,), float("inf"), **d)
    for i in range(4):
        z = h @ pn[f"w{i}"] + pn[f"b{i}"]
        margin = torch.minimum(margin, z.abs().min(dim=1).values)
        h = torch.relu(z)
    safe = torch.nonzero(margin > 2e-5)[:, 0]
    return traj, params, safe[torch.randperm(len(safe), generator=g, device=DEV)]


CFG = dict(clip_eps=0.2, ent_coef=0.01, vf_coef=0.5, illegal_l2_coef=0.0, value_clipping=True, reward_scaling=False,
           masked_policy=True)


def _ppo_reference(traj, params, idx, seed):
    """float64 autograd of the restated loss through the restated MLP on the device (as the existing parity test), with
    the minibatch's old log-probs / values / targets set near the current policy first (ratios straddle the clip range)"""
    from brl_b200.models import params_to_numpy
    from oracle import ppo_ref
    g = torch.Generator(device=DEV).manual_seed(seed)
    ref = {k: torch.tensor(v, dtype=torch.float64, device=DEV, requires_grad=True) for k, v in params_to_numpy(params).items()}
    hs, zs = [traj["obs"][idx].double()], []
    for i in range(4):
        z = hs[-1] @ ref[f"w{i}"] + ref[f"b{i}"]
        z.retain_grad()
        zs.append(z)
        hs.append(torch.relu(z))
    lg = hs[-1] @ ref["w4"] + ref["b4"]
    vl = (hs[-1] @ ref["w5"] + ref["b5"])[:, 0]
    lg.retain_grad()
    vl.retain_grad()
    mask, action, B = traj["mask"][idx], traj["action"][idx], len(idx)
    with torch.no_grad():
        ml = torch.where(mask, lg, torch.tensor(float("-inf"), dtype=torch.float64, device=DEV))
        lp_now = torch.log_softmax(ml, 1).gather(1, action.long()[:, None])[:, 0]
        traj["old_lp"][idx] = lp_now + (torch.rand(B, generator=g, dtype=torch.float64, device=DEV) - 0.5) * 0.8
        traj["old_v"][idx] = vl + torch.randn(B, generator=g, dtype=torch.float64, device=DEV) * 0.1
        traj["tgt"][idx] = vl + torch.randn(B, generator=g, dtype=torch.float64, device=DEV) * 0.2
    total_ref, aux = ppo_ref.loss_fn(lg, vl, mask, action, traj["old_lp"][idx], traj["old_v"][idx], traj["adv"][idx],
                                     traj["tgt"][idx], clip_eps=0.2, ent_coef=0.01, vf_coef=0.5)
    total_ref.backward()
    dzs = [z.grad for z in zs] + [lg.grad, vl.grad[:, None]]
    ins = hs[:4] + [hs[4], hs[4]]
    out = {"stats": np.array([float(total_ref.detach())] + [float(a.detach()) for a in aux])}
    for i in range(6):  # per element: the float64 gradient and sum |term| over the batch (the split's error scales with it)
        out[f"w{i}"] = (ref[f"w{i}"].grad.reshape(-1), (ins[i].detach().abs().T @ dzs[i].abs()).reshape(-1))
        out[f"b{i}"] = (ref[f"b{i}"].grad.reshape(-1), dzs[i].abs().sum(0).reshape(-1))
    return out


def _check_ppo(grads, stats, acc, want, what):
    """the bars of test_ppo_grad_matches_float64_autograd: loss scalars 5e-5, gradients 2e-4 of the tensor's largest +
    2e-5 of sum |term|, |grads|^2 in acc[14]; -> worst gradient error / bar"""
    np.testing.assert_allclose(stats.cpu().numpy()[:7], want["stats"], rtol=5e-5, atol=5e-6, err_msg=what)
    assert bool(torch.isfinite(grads).all()), f"{what}: a gradient element was not written"
    np.testing.assert_allclose(float(acc[14]), float((grads.double() ** 2).sum()), rtol=1e-5, err_msg=what)
    off, worst = 0, 0.0
    for k in [f"{c}{i}" for i in range(6) for c in ("w", "b")]:
        want_g, bound = want[k]
        got = grads[off:off + want_g.numel()].double()
        off += want_g.numel()
        r = float(((got - want_g).abs() / (2e-4 * want_g.abs().max() + 2e-5 * bound)).max())
        assert r <= 1.0, f"{what}: {k} {r:.3g} x the bar"
        worst = max(worst, r)
    assert off == grads.numel()
    return worst


def _ppo_call(traj, blob, scratch, idx, obs_dtype, tune):
    from brl_b200 import ops
    f32 = lambda t: t.to(torch.float32).contiguous()  # noqa: E731
    grads = torch.full((ops.mlp_num_params(),), float("nan"), dtype=torch.float32, device=DEV)
    stats = _nan(8)
    acc = ops.ppo_scratch(DEV).fill_(float("nan"))
    ops.ppo_grad(traj["obs"].to(obs_dtype).contiguous(), blob, scratch, idx.to(torch.int32), traj["mask"].to(torch.uint8).contiguous(),
                 traj["action"], f32(traj["old_lp"]), f32(traj["old_v"]), f32(traj["adv"]), f32(traj["tgt"]), grads, stats, acc,
                 tune=tune, **CFG)
    return grads, stats, acc


@pytest.mark.gpu
@pytest.mark.parametrize("tune,obs_dtype", [(0, torch.bfloat16), (4 | 16, torch.uint8)], ids=["tune0", "tune4|16"])
def test_ppo_grad_matches_float64_autograd_at_8205(tune, obs_dtype, record_property):
    """brl_ppo_grad at B = 8192 + 13 (65 row blocks, a ragged last one) on a poisoned scratch against float64 autograd"""
    from brl_b200 import ops
    from brl_b200.optim import flatten_params
    B = 8192 + 13
    traj, params, safe = _ppo_setup(20_000, seed=31)
    assert len(safe) >= B
    idx = safe[:B]
    want = _ppo_reference(traj, params, idx, seed=1)
    blob = ops.mlp_pack_train(flatten_params(params)[0])
    scratch = ops.mlp_train_scratch(B, DEV).fill_(0xFF)
    r = _check_ppo(*_ppo_call(traj, blob, scratch, idx, obs_dtype, tune), want, f"B={B} tune={tune}")
    record_property(f"ppo_grad B={B} tune={tune}", round(r, 4))


@pytest.mark.gpu
def test_ppo_grad_back_to_back_on_one_scratch(record_property):
    """two different minibatches (4109 and 1000 samples, disjoint rows) on one training scratch, no synchronisation in
    between, everything but the ABI's inputs poisoned first: each result matches its own float64 reference"""
    from brl_b200 import ops
    from brl_b200.optim import flatten_params
    B1, B2 = 4096 + 13, 1000
    traj, params, safe = _ppo_setup(10_000, seed=32)
    assert len(safe) >= B1 + B2
    idx1, idx2 = safe[:B1], safe[B1:B1 + B2]
    want1, want2 = _ppo_reference(traj, params, idx1, seed=2), _ppo_reference(traj, params, idx2, seed=3)
    blob = ops.mlp_pack_train(flatten_params(params)[0])
    scratch = ops.mlp_train_scratch(B1, DEV).fill_(0xFF)
    out1 = _ppo_call(traj, blob, scratch, idx1, torch.bfloat16, 0)
    out2 = _ppo_call(traj, blob, scratch, idx2, torch.bfloat16, 0)
    r = max(_check_ppo(*out1, want1, "first minibatch"), _check_ppo(*out2, want2, "second minibatch"))
    record_property("ppo_grad back-to-back", round(r, 4))
