"""Row-range sharded dense search on CPU: two and three gloo ranks running dense.ShardedIndexFlatL2's host logic
(range check, rank-major all-gather, global ids) with the oracle standing in for the CUDA local search and merge;
the merged lists must equal the single-index oracle bit for bit.  Also: pr_flat_merge's argument errors, the row
slice read_index(sharded=True) takes of a file, and the synth row-range generators."""
import ctypes
import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from flat_merge_oracle import merge_canonical
from oracle import flat_oracle as fo
from probing_rag_b200 import _lib, dense, sharding, synth

D_ = 64


def _matrix():
    """Every base row twice and a few three times, a block of zero rows: exact ties, across shard boundaries too."""
    rng = np.random.default_rng(11)
    base = rng.standard_normal((100, D_)).astype(np.float32)
    X = np.concatenate([base, base, np.zeros((20, D_), np.float32), base[:5]])
    Q = np.concatenate([base[:30], np.zeros((2, D_), np.float32), rng.standard_normal((4, D_)).astype(np.float32)])
    return X, Q


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded(X, rank, world, row_base=None, d=D_):
    lo, hi = sharding.shard_range(len(X), rank, world)
    Xl = X[lo:hi]

    def local_search(q, k):
        Dl, Il = fo.search_canonical(q.numpy(), Xl, k)
        return torch.from_numpy(Dl), torch.from_numpy(Il)

    def merge(gd, gi, bases):
        Dm, Im = merge_canonical(gd.numpy(), gi.numpy(), bases, gd.shape[2])
        return torch.from_numpy(Dm), torch.from_numpy(Im)

    shard = types.SimpleNamespace(d=d, ntotal=hi - lo)
    return dense.ShardedIndexFlatL2(shard, lo if row_base is None else row_base, local_search=local_search,
                                    merge=merge)


def _worker(rank, world, port, out_dir, path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        X, Q = _matrix()
        res = {}
        for name, rows in (("full", X), ("tiny", X[:4])):        # tiny: the last of three ranks holds no rows
            ix = _sharded(rows, rank, world)
            assert ix.ntotal == len(rows) and ix.d == D_ and ix.is_trained and ix.metric_type == 1
            for k in (5, 64):
                Dn, In = ix.search(Q, k)                          # NumPy in -> NumPy out
                assert isinstance(Dn, np.ndarray) and Dn.dtype == np.float32 and In.dtype == np.int64
                Dt, It = ix.search(torch.from_numpy(Q), k)        # tensor in -> tensor out
                assert isinstance(Dt, torch.Tensor) and np.array_equal(Dt.numpy(), Dn) and np.array_equal(It.numpy(), In)
                res[f"{name}_D{k}"], res[f"{name}_I{k}"] = Dn, In
            with pytest.raises(ValueError):
                ix.add(Q)
            with pytest.raises(ValueError):
                ix.reset()
        lo, hi = sharding.shard_range(len(X), rank, world)
        for bad in (dict(row_base=lo + (rank == 1)),              # gap before rank 1
                    dict(row_base=lo - (rank == 1)),              # rank 1 overlaps rank 0
                    dict(row_base=lo + 7),                        # does not start at 0
                    dict(d=D_ * 2 if rank == world - 1 else D_)):
            with pytest.raises(ValueError):                       # every rank sees the same ranges and raises
                _sharded(X, rank, world, **bad)
        base, mm = dense.read_shard_rows(path)
        assert base == lo and np.array_equal(np.asarray(mm), X[lo:hi])
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 3])
def test_row_shards_equal_single_index(tmp_path, world):
    X, Q = _matrix()
    path = str(tmp_path / "flat.index")
    dense.write_rows(path, X, D_)
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path), path), nprocs=world, join=True)
    for name, rows in (("full", X), ("tiny", X[:4])):
        for k in (5, 64):
            Dw, Iw = fo.search_canonical(Q, rows, k)
            for r in range(world):
                got = np.load(tmp_path / f"r{r}.npz")
                assert np.array_equal(got[f"{name}_I{k}"], Iw), f"rank {r} {name} k={k}: merged ids differ"
                assert np.array_equal(got[f"{name}_D{k}"], Dw), f"rank {r} {name} k={k}: merged distances differ"
    assert np.all(Iw[:, 4:] == -1)


def test_single_process_range_check():
    X, Q = _matrix()
    ix = _sharded(X, 0, 1)
    D, I = ix.search(Q, 10)
    Dw, Iw = fo.search_canonical(Q, X, 10)
    assert np.array_equal(D, Dw) and np.array_equal(I, Iw)
    with pytest.raises(ValueError, match="start at 0"):
        _sharded(X, 0, 1, row_base=3)


def test_merge_canonical_order_padding_and_bases():
    inf, fmax = np.float32(np.inf), fo.FLT_MAX
    D = np.array([[[0.5, 1.0, fmax]], [[0.5, inf, fmax]], [[0.25, 7.0, 9.0]]], np.float32)
    I = np.array([[[3, 1, -1]], [[0, 2, -1]], [[-1, 4, -1]]], np.int64)
    Dm, Im = merge_canonical(D, I, [0, 2 ** 33, 10], 6)
    assert Im.tolist() == [[3, 2 ** 33, 1, 14, 2 ** 33 + 2, -1]]
    assert Dm.tolist() == [[0.5, 0.5, 1.0, 7.0, float(inf), float(fmax)]]


def test_flat_merge_argument_errors_without_gpu():
    L = _lib.lib()
    p = ctypes.c_void_p(0x10000)
    base = (ctypes.c_int64 * 33)(*([0] * 33))
    assert L.pr_flat_merge(-1, 5, 2, p, p, base, p, p, None) == _lib.PR_EINVAL
    assert L.pr_flat_merge(4, 5, 0, p, p, base, p, p, None) == _lib.PR_EINVAL
    assert L.pr_flat_merge(4, 5, 33, p, p, base, p, p, None) == _lib.PR_EINVAL
    assert b"n_lists" in L.pr_last_error()
    assert L.pr_flat_merge(4, 0, 2, p, p, base, p, p, None) == _lib.PR_EINVAL
    assert L.pr_flat_merge(4, 129, 2, p, p, base, p, p, None) == _lib.PR_EINVAL
    assert b"k must be" in L.pr_last_error()
    for i in range(4):
        ptrs = [p] * 4
        ptrs[i] = None
        assert L.pr_flat_merge(4, 5, 2, ptrs[0], ptrs[1], base, ptrs[2], ptrs[3], None) == _lib.PR_EINVAL
    assert L.pr_flat_merge(4, 5, 2, p, p, None, p, p, None) == _lib.PR_EINVAL
    neg = (ctypes.c_int64 * 2)(0, -5)
    assert L.pr_flat_merge(4, 5, 2, p, p, neg, p, p, None) == _lib.PR_EINVAL
    assert b"negative" in L.pr_last_error()
    assert L.pr_flat_merge(0, 5, 2, None, None, base, None, None, None) == _lib.PR_OK     # nothing to merge


def test_synth_row_ranges_and_queries(monkeypatch):
    monkeypatch.setattr(synth, "EMB_BLOCK", 1000)
    n, d = 3500, 64
    for kind in ("clustered", "isotropic"):
        full = synth.dense_rows(n, d, device="cpu", kind=kind)
        for lo, hi in ((0, n), (0, 0), (999, 1001), (1000, 2000), (1234, 3500), (3499, 3500), (3500, 3500)):
            assert torch.equal(synth.dense_rows(n, d, device="cpu", kind=kind, row_lo=lo, row_hi=hi), full[lo:hi])
        for B in (1, 37):
            assert torch.equal(synth.dense_queries_of(n, d, B, device="cpu", kind=kind), synth.dense_queries(full, B))
    with pytest.raises(ValueError):
        synth.dense_rows(n, d, device="cpu", row_lo=10, row_hi=5)
