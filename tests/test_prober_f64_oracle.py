"""The float64 prober restatement and the pooling restatement (tests/prober_f64_oracle.py) against the fp32 oracle
and the golden outputs of the reference's own ImprovedProbe (CPU)."""
import os

import numpy as np
import torch

from oracle import prober_oracle as po
import prober_f64_oracle as pf
from test_prober_oracle import GOLDEN_THREADS, load_probers


def test_f64_restatement_matches_the_fp32_oracle_and_the_golden_outputs(golden_dir):
    g = np.load(os.path.join(golden_dir, "prober_golden.npz"))
    x = po.make_hidden_states(int(g["n"]), seed=0)
    sds64 = [pf.state_f64(po.make_prober_state(layer)) for layer in po.PROBE_LAYERS]
    n_threads = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        ref32 = po.prober_logits(load_probers(), x)
        l64 = pf.prober_logits_f64(sds64, x)
    finally:
        torch.set_num_threads(n_threads)
    assert l64.dtype == torch.float64 and l64.shape == ref32.shape
    # the fp32 module is off the exact value by its own rounding (2048-long f32 sums): ~1e-5 on logits of std ~3
    assert (l64 - ref32.double()).abs().max().item() < 2e-5
    assert (l64 - torch.from_numpy(g["logits"]).double()).abs().max().item() < 2e-5
    probs, psum, _ = pf.gate_f64(l64)
    assert (probs - torch.softmax(ref32.double(), -1)).abs().max().item() < 1e-5
    assert np.abs(psum.numpy() - g["probsum"]).max() < 1e-5
    for j, th in enumerate(g["thetas"]):
        _, psum, ret = pf.gate_f64(l64, float(th))
        margin = np.abs(g["probsum"][:, 0] + float(th) - g["probsum"][:, 1])
        assert np.all((ret.numpy() == g["retrieve"][j]) | (margin < 1e-5))


def test_f64_gate_ablation_and_failed_comparisons():
    logits = torch.tensor([[[0.0, 1.0], [2.0, -1.0]],
                           [[float("nan"), 0.0], [0.0, 0.0]],
                           [[float("inf"), 0.0], [0.0, 0.0]]], dtype=torch.float64)
    probs, psum, ret = pf.gate_f64(logits, 0.0, 0)
    assert torch.allclose(psum[0], probs[0].sum(0))
    assert ret.tolist() == [True, True, True]             # NaN sums: P0 + theta < P1 is False -> retrieve
    _, psum, ret = pf.gate_f64(logits, 0.0, 1)             # only prober 1
    assert torch.equal(psum[0], probs[0, 1])
    _, psum, ret = pf.gate_f64(logits, -0.5, 2)            # ablation == P: empty sum, retrieve = NOT (theta < 0)
    assert torch.equal(psum, torch.zeros(3, 2, dtype=torch.float64)) and not bool(ret.any())
    _, _, ret = pf.gate_f64(logits, 0.0, 2)
    assert bool(ret.all())


def test_pool_restatement_sums_tokens_in_order_then_adds_once():
    # f32 order matters: (1e8 + 1) + -1e8 = 0 in token order, and the call's sum is added to the accumulator once
    act = np.array([[[1e8], [1.0], [-1e8], [0.25]]], dtype=np.float32).repeat(4, axis=2)
    acc = np.full((2, 3, 4), 0.5, dtype=np.float32)
    pf.pool_call(acc, 1, act)
    assert np.array_equal(acc[0, 1], np.full(4, 0.75, np.float32))
    assert np.array_equal(acc[1], np.full((3, 4), 0.5, np.float32)) and np.array_equal(acc[0, 0], acc[0, 2])
    acc = np.zeros((1, 1, 4), dtype=np.float32)
    pf.pool_call(acc, 0, np.array([[[3e7], [1.0], [1.0]]], dtype=np.float32).repeat(4, axis=2))
    assert acc[0, 0, 0] == np.float32(3e7) + np.float32(1.0) + np.float32(1.0)   # not 3e7 + 2
    # row_map: negative entries skip the row
    rng = np.random.default_rng(0)
    act = rng.standard_normal((3, 5, 8)).astype(np.float32)
    acc = np.zeros((4, 2, 8), dtype=np.float32)
    pf.pool_call(acc, 0, act, row_map=[3, -1, 0])
    s = act.sum(axis=1, dtype=np.float64)
    assert np.allclose(acc[3, 0], s[0], atol=1e-5) and np.allclose(acc[0, 0], s[2], atol=1e-5)
    assert not acc[1].any() and not acc[2].any() and not acc[:, 1].any()
