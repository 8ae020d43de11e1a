"""Prober oracle against the golden outputs of the reference's own ImprovedProbe (CPU)."""
import hashlib
import os

import numpy as np
import torch

from oracle import prober_oracle as po

# The golden logits are float32 CPU matmuls whose summation order depends on the number of intra-op threads (the
# BLAS splits the 2048-long reductions differently, ~5e-6 apart).  They were written with this many threads; with it
# the oracle reproduces them bit for bit whatever the host's core count.
GOLDEN_THREADS = 8


def load_probers():
    probers = []
    for layer in po.PROBE_LAYERS:
        p = po.OracleImprovedProbe(po.D_MODEL, po.N_CLASSES)
        p.load_state_dict(po.make_prober_state(layer))
        probers.append(p.eval())
    return probers


def test_oracle_matches_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, "prober_golden.npz"))
    x = po.make_hidden_states(int(g["n"]), seed=0)
    assert hashlib.sha256(x.numpy().tobytes()).hexdigest() == str(g["x_digest"])
    for layer, dig in zip(po.PROBE_LAYERS, g["state_digests"]):
        assert po.state_digest(po.make_prober_state(layer)) == str(dig)
    n_threads = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        logits = po.prober_logits(load_probers(), x)
    finally:
        torch.set_num_threads(n_threads)
    assert np.allclose(logits.numpy(), g["logits"], rtol=1e-5, atol=1e-6)
    for j, th in enumerate(g["thetas"]):
        psum, ret = po.gate(torch.from_numpy(g["logits"]), float(th), 0)
        if j == 0:
            assert np.allclose(psum.numpy(), g["probsum"], atol=1e-6)
        assert np.array_equal(ret.numpy(), g["retrieve"][j])


def test_param_count_and_state_keys():
    p = po.OracleImprovedProbe(2048, 2)
    assert sum(t.numel() for t in p.parameters()) == 1318914      # exp_parameter_check.py:52
    assert set(p.state_dict().keys()) == set(po.STATE_KEYS)


def test_pooling_and_round_control():
    cache = [torch.ones(1, 7, 4), torch.full((1, 1, 4), 2.0), torch.full((1, 1, 4), 3.0)]
    assert torch.equal(po.pool_hidden_states(cache), torch.full((1, 4), 5.0))   # prefill dropped, SUM
    assert po.retrieval_rounds([False]) == 0
    assert po.retrieval_rounds([True, False]) == 1
    assert po.retrieval_rounds([True, True, True, False]) == 3
    assert po.retrieval_rounds([True] * 6) == 4                                  # cap: exp_rag.py:462-465
