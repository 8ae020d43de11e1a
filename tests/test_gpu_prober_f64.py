"""The fused prober (csrc/prober.cu) and the pooler (csrc/pool.cu) against float64 / exact restatements
(tests/prober_f64_oracle.py), over the whole input domain the kernels accept.

test_gpu_prober.py holds the kernel to the 1e-3 bar on probabilities against the fp32 module.  Here the logits and
probabilities are held to bounds measured on the B200 with about 4x headroom (DESIGN §4.3): a saturated softmax hides a
logit error of 0.1 from a probability check, a logit check does not.  Invariants that hold by construction (a row's
result does not depend on its neighbours, its position, the other probers or the logits output) are asserted bit for
bit, and the pooler is asserted bit for bit against its promise."""
import functools
import math

import numpy as np
import pytest
import torch

import prober_f64_oracle as pf
from oracle import prober_oracle as po

pytestmark = pytest.mark.gpu

# Error bounds against the float64 reference (DESIGN §4.3): max |logit - logit_f64| and max |p - p_f64| over the
# probers, max |probsum - probsum_f64|.  The worst over this file's inputs on a B200 (1,000 W) was 9.3e-5 / 3.1e-5 /
# 4.5e-5; the bounds leave 3-4x headroom.
LOGIT_TOL = 4e-4
PROB_TOL = 1e-4
PSUM_TOL = 2e-4

D_MODELS = (128, 384, 640, 1152, 1920, 2048)
NS = (1, 127, 128, 129, 255, 256, 257, 511, 512, 513, 4097)
X_DTYPES = (torch.float32, torch.bfloat16, torch.float16)
PAIR = 256                         # rows of one CTA pair

worst = {"logit": 0.0, "prob": 0.0, "probsum": 0.0}


@pytest.fixture(scope="module", autouse=True)
def report_worst():
    yield
    print(f"\nworst errors against the float64 reference: {worst}")


@functools.lru_cache(maxsize=2)
def gate_of(P, d_model):
    """(ProberGate, state_dicts in f64) of P synthetic probers; prober i is make_prober_state(6 + 2 i)."""
    from probing_rag_b200.prober import ProberGate
    sds = [po.make_prober_state(6 + 2 * i, d_model=d_model) for i in range(P)]
    return ProberGate(sds, device="cuda"), [pf.state_f64(sd) for sd in sds]


def hidden(n, P, d_model, seed):
    """f32 [n, P, d] on the device: s * Normal(0, 1) with a per-row scale s ~ LogUniform(10, 300), the pooled hidden
    states of synth.make_hidden_states, generated on the device."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(n, P, d_model, device="cuda", generator=g)
    s = torch.empty(n, 1, 1, device="cuda").uniform_(math.log(10.0), math.log(300.0), generator=g).exp()
    return x * s


def sample_rows(n, seed, extra=32):
    """The first and last row of every CTA pair plus a seeded random set."""
    rows = {0, n - 1}
    for b in range(0, n, PAIR):
        rows.update((b, min(b + PAIR - 1, n - 1)))
    rows.update(np.random.default_rng(seed).integers(0, n, size=min(extra, n)).tolist())
    return torch.tensor(sorted(rows))


def check_f64(out, x, sds64, rows=None, theta=0.0, ablation=0):
    """out (want_logits=True) against the float64 reference on `rows` of x (all rows if None)."""
    rows = torch.arange(x.shape[0]) if rows is None else rows
    l64 = pf.prober_logits_f64(sds64, x[rows.to(x.device)].cpu())
    p64, ps64, _ = pf.gate_f64(l64, theta, ablation)
    lg = out.logits.cpu()[rows].double()
    ps = out.probsum.cpu()[rows].double()
    assert bool(torch.isfinite(lg).all()) and bool(torch.isfinite(l64).all())
    dl = (lg - l64).abs().amax(dim=(0, 2))
    dp = (torch.softmax(lg, -1) - p64).abs().amax(dim=(0, 2))
    dps = (ps - ps64).abs().max().item()
    worst["logit"] = max(worst["logit"], dl.max().item())
    worst["prob"] = max(worst["prob"], dp.max().item())
    worst["probsum"] = max(worst["probsum"], dps)
    assert dl.max().item() < LOGIT_TOL, f"max |logit - f64| per prober {dl.tolist()}"
    assert dp.max().item() < PROB_TOL, f"max |p - f64| per prober {dp.tolist()}"
    assert dps < PSUM_TOL, dps
    check_decisions(out, theta)


def check_decisions(out, theta):
    """retrieve == NOT (double(p0) + theta < double(p1)) on the kernel's own probsum; retrieve_idx its nonzero rows."""
    p = out.probsum.cpu().double()
    want = ~(p[:, 0] + theta < p[:, 1])
    assert torch.equal(out.retrieve.cpu(), want)
    assert torch.equal(out.retrieve_idx.cpu().long(), torch.nonzero(want).flatten())
    assert int(out.n_retrieve.item()) == int(want.sum())


# ---- accuracy over the shape grid --------------------------------------------------------------------------------
def test_default_workload_error_bounds():
    """The benchmark's workload: 16,384 rows x 6 probers x 2048 features (tools/bench_prober.py)."""
    gate, sds64 = gate_of(6, 2048)
    x = po.make_hidden_states(16384, seed=4).cuda()
    out = gate(x, want_logits=True)
    check_f64(out, x, sds64, rows=sample_rows(16384, seed=4, extra=1024))


@pytest.mark.parametrize("d_model", D_MODELS)
@pytest.mark.parametrize("P", range(1, 9))
def test_shape_grid_against_f64(P, d_model):
    """P = 1..8, d_model from one k-block pair (128: n_iter == kStages) to 2048 through non-powers of two; n around
    the CTA and pair boundaries; f32 / bf16 / f16 inputs; ablation 0, 1, P - 1, P (P: the empty sum)."""
    gate, sds64 = gate_of(P, d_model)
    ablations = sorted({0, 1, P - 1, P})
    for i, n in enumerate(NS):
        x32 = hidden(n, P, d_model, seed=1000 * P + d_model + n)
        rows = sample_rows(n, seed=n)
        for dtype in X_DTYPES:
            x = x32.to(dtype)
            outs = [gate(x, theta=0.05 * (a - 1), ablation=a, want_logits=True) for a in ablations]
            for a, out in zip(ablations, outs):
                assert torch.equal(out.logits, outs[0].logits)          # the gate does not touch the logits
                check_f64(out, x, sds64, rows, theta=0.05 * (a - 1), ablation=a)
            empty = outs[-1]                                             # ablation == P
            assert not bool(empty.probsum.any())
            assert bool(empty.retrieve.all()) == (0.05 * (P - 1) >= 0)


# ---- bit-exact invariants ----------------------------------------------------------------------------------------
def test_a_row_does_not_depend_on_its_neighbours_or_position():
    gate, _ = gate_of(6, 2048)
    x = hidden(4097, 6, 2048, seed=1)
    full = gate(x, want_logits=True).logits
    rows = (0, 1, 127, 128, 255, 256, 300, 511, 512, 4095, 4096)
    for r in rows:
        assert torch.equal(gate(x[r:r + 1], want_logits=True).logits[0], full[r]), r
    y = hidden(600, 6, 2048, seed=2)
    for pos in (0, 127, 128, 255, 256, 599):
        z = y.clone()
        z[pos] = x[300]
        assert torch.equal(gate(z, want_logits=True).logits[pos], full[300]), pos
    # rows holding NaN / inf retrieve (the reference's comparison fails) and change no other row
    z = x[:513].clone()
    bad = {0: ("nan", None), 5: ("nan", 7), 255: ("inf", 2000), 256: ("-inf", 64), 257: ("inf", 0), 512: ("nan", 2047)}
    for r, (v, f) in bad.items():
        if f is None:
            z[r] = float(v)
        else:
            z[r, :, f] = float(v)
    out = gate(z, want_logits=True)
    good = torch.tensor([r for r in range(513) if r not in bad])
    assert torch.equal(out.logits[good.cuda()], full[:513][good.cuda()])
    assert bool(out.retrieve[list(bad)].all())
    assert not bool(torch.isfinite(out.probsum[list(bad)]).any())
    assert set(bad) <= set(out.retrieve_idx.tolist())
    check_decisions(out, 0.0)


def test_a_prober_does_not_depend_on_the_others():
    from probing_rag_b200.prober import ProberGate
    gate, _ = gate_of(8, 640)
    x = hidden(513, 8, 640, seed=3)
    full = gate(x, want_logits=True).logits
    for p in range(8):
        one = ProberGate([po.make_prober_state(6 + 2 * p, d_model=640)], device="cuda")
        assert torch.equal(one(x[:, p:p + 1], want_logits=True).logits[:, 0], full[:, p]), p


@pytest.mark.parametrize("n", [1, 257, 4097])
def test_the_logits_output_does_not_change_the_result(n):
    gate, _ = gate_of(6, 2048)
    x = hidden(n, 6, 2048, seed=n)
    for kw in (dict(), dict(theta=0.1, ablation=2), dict(sync=False)):
        a = gate(x, want_logits=True, **kw)
        b = gate(x, want_logits=False, **kw)
        assert b.logits is None
        for f in ("probsum", "retrieve", "retrieve_idx", "n_retrieve"):
            assert torch.equal(getattr(a, f), getattr(b, f)), (kw, f)


# ---- gate and compaction at scale --------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 255, 256, 257, 65537, (1 << 20) + 3])
def test_gate_and_compaction_at_scale(n):
    """P = 1, d_model = 128 keeps X small; 2^20 + 3 rows are 4,097 compaction blocks."""
    gate, _ = gate_of(1, 128)
    x = hidden(n, 1, 128, seed=7)
    base = gate(x)
    p = base.probsum.cpu().double()
    gap = (p[:, 1] - p[:, 0]).sort().values
    thetas = (0.0, float(gap[n // 2]), float(gap[n // 3]), -2.0, 2.0)   # about half / a third / no row / every row
    for theta in thetas:
        for sync in (True, False):
            out = gate(x, theta=theta, sync=sync)
            assert torch.equal(out.probsum, base.probsum)
            want = ~(p[:, 0] + theta < p[:, 1])
            assert torch.equal(out.retrieve.cpu(), want)
            idx = torch.nonzero(want).flatten()
            k = int(out.n_retrieve.item())
            assert k == idx.numel()
            got = out.retrieve_idx.cpu().long()
            if sync:
                assert torch.equal(got, idx)
            else:
                assert got.shape == (n,) and torch.equal(got[:k], idx) and bool((got[k:] == -1).all())
        if theta == -2.0:
            assert k == 0
        if theta == 2.0:
            assert k == n
    out = gate(x, theta=0.0, ablation=1, sync=False)         # the empty sum: 0 + 0 < 0 is False, every row retrieves
    assert not bool(out.probsum.any()) and int(out.n_retrieve.item()) == n
    assert torch.equal(out.retrieve_idx.cpu().long(), torch.arange(n))


# ---- input sweep -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ratio", [0, 10, 100, 300, 1000, 3000])
def test_common_offset_against_f64(ratio):
    """x = sigma * Normal(0, 1) + c with |c| = ratio * sigma.  The input LayerNorm is folded around fc1, and the bf16
    split of x is relative to |x|: unless the kernel subtracts a per-row shift first, the error grows like |c| / sigma."""
    gate, sds64 = gate_of(6, 2048)
    sigma = 50.0
    x = hidden(512, 6, 2048, seed=ratio)
    x = x / x.std(dim=-1, keepdim=True) * sigma
    sign = torch.where(torch.arange(512, device="cuda") % 2 == 0, 1.0, -1.0)[:, None, None]
    x = x + sign * (ratio * sigma)
    check_f64(gate(x, want_logits=True), x, sds64)


def test_special_rows_against_f64():
    """Constant rows (sigma = 0: LN_in gives beta exactly), zero rows, rows with a few massive features, tiny and huge
    scales, next to ordinary rows."""
    gate, sds64 = gate_of(6, 2048)
    x = hidden(640, 6, 2048, seed=9)
    g = torch.Generator(device="cuda").manual_seed(10)
    for i, c in enumerate((1.0, -3.5, 0.1, 1e3, -7e4, 123.456)):
        x[i] = c
    x[6:10] = 0.0
    for j, r in enumerate(range(10, 90)):                 # 1 to 4 features 1000x the rest, in any k-block
        feats = torch.randint(0, 2048, (1 + j % 4,), device="cuda", generator=g)
        x[r, :, feats] = x[r, :, feats].sign() * 1000.0 * x[r].abs().amax()
    x[90:150] *= 1e-3 / x[90:150].std(dim=-1, keepdim=True)
    x[150:210] *= 1e4 / x[150:210].std(dim=-1, keepdim=True)
    x[210:260] = x[210:260] / x[210:260].std(dim=-1, keepdim=True) * 50.0 + 1e4   # huge scale, large offset
    check_f64(gate(x, want_logits=True), x, sds64)


def test_f16_inputs_near_the_f16_maximum():
    gate, sds64 = gate_of(6, 2048)
    x = hidden(257, 6, 2048, seed=12)
    x = (x / x.abs().amax(dim=-1, keepdim=True) * 65504.0).clamp(-65504.0, 65504.0)
    x[::3, :, 5] = 65504.0
    x[1::3, :, 1000] = -65504.0
    xh = x.to(torch.float16)
    assert bool(torch.isfinite(xh).all())
    out = gate(xh, want_logits=True)
    check_f64(out, xh, sds64)
    assert torch.equal(gate(xh.float(), want_logits=True).logits, out.logits)


# ---- pooler ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d_model", [4, 12, 516, 2052])
@pytest.mark.parametrize("dtype", X_DTYPES)
def test_pooler_bit_exact_against_the_restatement(dtype, d_model):
    """d_model / 4 not a multiple of 128 leaves a partial block; 1 to 1,000 tokens per call; contiguous, zero (expanded)
    and padded token strides, padded row strides; a row_map that skips rows.  Every call sums its tokens in fp32 in
    token order from 0 and adds the sum once: the accumulator must equal the restatement bit for bit."""
    from probing_rag_b200.pooling import HiddenStatePooler
    g = torch.Generator(device="cuda").manual_seed(d_model)
    n_rows, layers = 6, ["a", "b", "c"]
    pooler = HiddenStatePooler(n_rows, layers, d_model)
    ref = np.zeros((n_rows, len(layers), d_model), dtype=np.float32)

    def act(R, T, pad_tok=0):
        a = torch.randn(R, T, d_model + pad_tok, device="cuda", generator=g) * 3.0
        return a.to(dtype)[:, :, :d_model]

    calls = [
        ("a", act(6, 1), None),
        ("b", act(6, 7), None),
        ("c", act(4, 1000), torch.tensor([5, -1, 0, 2], dtype=torch.int32)),
        ("a", act(6, 64, pad_tok=8), None),                                     # padded token stride
        ("b", act(6, 5, pad_tok=4)[::2], torch.tensor([1, 3, -7], dtype=torch.int32)),   # padded row stride
        ("c", act(6, 1).expand(6, 333, d_model), None),                         # zero token stride
        ("b", act(2, 1000)[:, ::2], torch.tensor([-1, 4], dtype=torch.int32)),  # every other token
    ]
    for layer, a, rm in calls:
        pooler.add(layer, a, row_map=rm)
        pf.pool_call(ref, layers.index(layer), a.float().cpu().numpy(), None if rm is None else rm.numpy())
        torch.cuda.synchronize()
        assert np.array_equal(pooler.X.cpu().numpy(), ref), (layer, tuple(a.shape), a.stride())
    assert calls[5][1].stride(1) == 0


def test_pooler_row_map_contract():
    """Non-negative row_map entries must be distinct and inside the accumulator; negative entries skip the row.  Two
    rows into one accumulator row would race, so add() refuses the map before anything runs."""
    from probing_rag_b200.pooling import HiddenStatePooler
    pooler = HiddenStatePooler(4, ["a"], 8)
    a = torch.ones(3, 2, 8, device="cuda")
    for bad in ([0, 0, 1], [1, -1, 1], [0, 4, 1], [0, 1, 2 ** 31], [0, 1]):
        with pytest.raises(ValueError):
            pooler.add("a", a, row_map=torch.tensor(bad, dtype=torch.int64))
    torch.cuda.synchronize()
    assert not bool(pooler.X.any())
    pooler.add("a", a, row_map=torch.tensor([3, -1, -5], dtype=torch.int32, device="cuda"))
    want = torch.zeros(4, 1, 8)
    want[3] = 2.0
    assert torch.equal(pooler.X.cpu(), want)
