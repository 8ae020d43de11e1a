"""IndexFlatL2 / IndexFlatIP.add copies the rows, as faiss does, and a search on a second GPU of the process launches as
on the first.  Every comparison is against a clone of the rows taken at add time, never against index.rows()."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

from oracle import flat_ip_oracle as fio
from oracle import flat_oracle as fo
from probing_rag_b200 import IndexFlatIP, IndexFlatL2, ShardedIndexFlatL2, synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _same(got, want):
    D, I = got
    Dr, Ir = want
    return np.array_equal(I.cpu().numpy(), Ir) and np.array_equal(D.cpu().numpy().view(np.uint32), Dr.view(np.uint32))


def _canonical(cls, Q, X, k):
    return fo.search_canonical_torch(Q, X, k) if cls is IndexFlatL2 else fio.search_canonical_ip_torch(Q, X, k)


@pytest.mark.parametrize("cls", [IndexFlatL2, IndexFlatIP])
def test_a_reused_buffer_keeps_every_batch(cls):
    rows = synth.dense_rows(12_000, 256)
    buf = torch.empty((4000, 256), device="cuda")
    index = cls(256)
    for a in range(0, 12_000, 4000):
        buf.copy_(rows[a:a + 4000])
        index.add(buf)
    buf.zero_()
    assert index.ntotal == 12_000 and torch.equal(index.rows(), rows)
    Q = synth.dense_queries(rows, 17)
    assert _same(index.search(Q, 10), _canonical(cls, Q, rows, 10))


@pytest.mark.parametrize("cls", [IndexFlatL2, IndexFlatIP])
def test_changing_the_added_tensor_after_a_search_changes_nothing(cls):
    rows = synth.dense_rows(20_000, 128)
    kept = rows.clone()
    index = cls(128)
    index.add(rows)
    Q = synth.dense_queries(kept, 33)
    want = _canonical(cls, Q, kept, 10)
    assert _same(index.search(Q, 10), want)
    rows.mul_(-3.0).add_(1.0)                      # the filter's bf16 copy and the exact rows must both stay
    assert _same(index.search(Q, 10), want)
    assert torch.equal(index.rows(), kept)


def test_sharded_index_at_world_one():
    rows = synth.dense_rows(20_000, 128)
    kept = rows.clone()
    shard = IndexFlatL2(128)
    shard.add(rows)
    sx = ShardedIndexFlatL2(shard, 0)
    Q = synth.dense_queries(kept, 9)
    want = fo.search_canonical_torch(Q, kept, 10)
    assert _same(sx.search(Q, 10), want)
    rows.zero_()
    assert _same(sx.search(Q, 10), want)


_TWO_DEVICES = textwrap.dedent("""
    import numpy as np, torch
    from oracle import flat_oracle as fo, flat_ip_oracle as fio, prober_oracle as po
    from probing_rag_b200 import IndexFlatIP, IndexFlatL2, synth
    from probing_rag_b200.prober import ProberGate
    probers = []
    for layer in po.PROBE_LAYERS:
        p = po.OracleImprovedProbe(po.D_MODEL, po.N_CLASSES)
        p.load_state_dict(po.make_prober_state(layer))
        probers.append(p.eval())
    x = po.make_hidden_states(300, seed=5)
    ref = torch.softmax(po.prober_logits(probers, x), -1)
    for dev in ("cuda:0", "cuda:1"):
        rows = synth.dense_rows(30_000, 768, device=dev)
        Q = synth.dense_queries(rows, 40)
        for cls, canon in ((IndexFlatL2, fo.search_canonical_torch), (IndexFlatIP, fio.search_canonical_ip_torch)):
            index = cls(768, dev)
            index.add(rows)
            D, I = index.search(Q, 10)
            Dr, Ir = canon(Q, rows, 10)
            assert np.array_equal(I.cpu().numpy(), Ir), (dev, cls.__name__)
            assert np.array_equal(D.cpu().numpy().view(np.uint32), Dr.view(np.uint32)), (dev, cls.__name__)
        gate = ProberGate([p.state_dict() for p in probers], device=dev)
        out = gate(x.to(dev), want_logits=True)
        err = (torch.softmax(out.logits.cpu(), -1) - ref).abs().max().item()
        assert err < 1e-3, (dev, err)
        print(dev, "ok", flush=True)
""")


@pytest.mark.timeout(600)
def test_search_and_prober_on_a_second_device_of_the_process():
    """A fresh process runs IndexFlatL2, IndexFlatIP and ProberGate on cuda:0, then on cuda:1: the kernels' dynamic
    shared memory attribute has to hold on each device."""
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, this box has {torch.cuda.device_count()}")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests")]))
    res = subprocess.run([sys.executable, "-c", _TWO_DEVICES], cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=540)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "cuda:1 ok" in res.stdout
