"""Row-range sharded exact dense search on the GPU: pr_flat_merge against its CPU restatement, shards simulated on one
device against the single index, and one process per GPU over NCCL (read_index(sharded=True)) against the single
index and the oracle -- ids AND distances bit for bit."""
import os
import socket

import numpy as np
import pytest
import torch

from flat_merge_oracle import merge_canonical
from oracle import flat_oracle as fo
from probing_rag_b200 import IndexFlatL2, ShardedIndexFlatL2, dense, read_index, sharding, synth, write_index
from test_gpu_flat import SHAPES

pytestmark = pytest.mark.gpu

FMAX = float(np.finfo(np.float32).max)


# ---------------------------------------------------------------------------------------------- pr_flat_merge
def _lists(rng, L, B, k, short="some", empty_list=False):
    """[L, B, k] ranked lists as pr_flat_search writes them: distances from a small set (exact ties within and
    across lists, real FLT_MAX, +inf and NaN), distinct local ids per list, (distance bits, id) ascending with NaN
    as 0x7FFFFFFF after +inf, padded tails whose distance is arbitrary.  A NaN is then given one of several bit
    patterns (either sign, other payloads): the merge ranks and returns every NaN as 0x7FFFFFFF."""
    values = np.array([0.0, 0.25, 0.5, 1.0, 1.0 + 2 ** -23, 3.0, FMAX, np.inf, np.nan], np.float32)
    dist_ = rng.choice(values, size=(L, B, k)).astype(np.float32)
    dist_[np.isnan(dist_)] = np.uint32(0x7FFFFFFF).view(np.float32)
    ids = np.argsort(rng.random((L, B, 3 * k)), axis=-1)[:, :, :k].astype(np.int64)
    m = rng.integers(0, k + 1, size=(L, B)) if short == "some" else \
        (rng.integers(0, k, size=(L, B)) if short == "all" else np.full((L, B), k))
    if empty_list:
        m[0] = 0
    pad = np.arange(k)[None, None, :] >= m[:, :, None]
    key = (dist_.view(np.uint32).astype(np.uint64) << np.uint64(32)) | ids.astype(np.uint64)
    key[pad] = np.iinfo(np.uint64).max
    key.sort(axis=-1)
    pad = key == np.iinfo(np.uint64).max
    dist_ = (key >> np.uint64(32)).astype(np.uint32).view(np.float32)
    ids = (key & np.uint64(0xFFFFFFFF)).astype(np.int64)
    nan = np.isnan(dist_)
    dist_[nan] = rng.choice(np.array([0x7FFFFFFF, 0x7FC00000, 0xFFC00000, 0x7FC0BEEF, 0xFFFFFFFF], np.uint32),
                            size=int(nan.sum())).view(np.float32)
    dist_[pad] = rng.choice(np.array([FMAX, 0.0, 2.0, np.nan], np.float32), size=int(pad.sum()))
    ids[pad] = -1
    return dist_, ids


MERGE_CASES = [  # (lists, k, B, rows short of k, an all-padding list, bases)
    (1, 1, 1, "some", False, "big"), (1, 128, 64, "none", False, "big"), (2, 5, 65536, "some", False, "big"),
    (3, 100, 257, "all", False, "big"), (8, 128, 1000, "some", True, "big"), (32, 128, 300, "some", False, "big"),
    (32, 1, 513, "none", True, "big"), (16, 5, 4096, "all", False, "zero"), (5, 10, 2000, "some", True, "zero"),
]


@pytest.mark.parametrize("L, k, B, short, empty_list, bases", MERGE_CASES)
def test_merge_against_oracle(L, k, B, short, empty_list, bases):
    rng = np.random.default_rng(L * 1000 + k * 7 + B)
    Dl, Il = _lists(rng, L, B, k, short, empty_list)
    # "big": ranges above 2^32 (ids compared as 64 bits); "zero": every list at base 0, so equal global ids tie
    # across lists and rank in list order
    base = [int(b) for b in np.sort(rng.integers(0, 2 ** 40, size=L)) + 2 ** 32] if bases == "big" else [0] * L
    D, I = dense.merge_lists(torch.from_numpy(Dl).cuda(), torch.from_numpy(Il).cuda(), base)
    Dw, Iw = merge_canonical(Dl, Il, base, k)
    assert np.array_equal(I.cpu().numpy(), Iw)
    assert np.array_equal(D.cpu().numpy().view(np.uint32), Dw.view(np.uint32))


# ---------------------------------------------------------------------------------------------- simulated shards
def _split(n, parts):
    """shard_range's cut of [0, n) into `parts`, with an extra empty range after the first."""
    r = [sharding.shard_range(n, i, parts) for i in range(parts)]
    return [r[0], (r[0][1], r[0][1])] + r[1:]


def _same_bits(a, b):
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


def _check_shards(rows, Q, k):
    single = IndexFlatL2(rows.shape[1])
    single.add(rows)
    Ds, Is = single.search(Q, k)
    for parts in (2, 3, 8):
        ranges = _split(rows.shape[0], parts)
        Dl, Il = [], []
        for lo, hi in ranges:
            sh = IndexFlatL2(rows.shape[1])
            sh.add(rows[lo:hi])
            d, i = sh.search(Q, k)
            Dl.append(d)
            Il.append(i)
        D, I = dense.merge_lists(torch.stack(Dl), torch.stack(Il), [lo for lo, _ in ranges])
        assert torch.equal(I, Is) and _same_bits(D, Ds), f"{parts} shards differ from the single index"
    sx = ShardedIndexFlatL2(single, 0)                   # world 1 (no process group): the full path
    D, I = sx.search(Q, k)
    assert sx.ntotal == rows.shape[0] and torch.equal(I, Is) and _same_bits(D, Ds)
    return Ds, Is


@pytest.mark.parametrize("n, d, B, k", SHAPES)
def test_simulated_shards_equal_single_index(n, d, B, k):
    rows = synth.dense_rows(n, d)
    _check_shards(rows, synth.dense_queries(rows, B), k)


def test_simulated_shards_isotropic_and_ties():
    rows = synth.dense_rows(100_003, 768, kind="isotropic")
    _check_shards(rows, synth.dense_queries(rows, 64), 10)
    g = torch.Generator(device="cuda").manual_seed(5)
    base = torch.randn((300, 128), generator=g, device="cuda")
    X = torch.cat([base, base, torch.zeros((40, 128), device="cuda"), base[:5]])   # exact ties across every cut
    Q = torch.cat([base[:20], torch.zeros((3, 128), device="cuda")])
    D, I = _check_shards(X, Q, 64)
    Dr, Ir = fo.search_canonical_torch(Q, X, 64)
    assert np.array_equal(I.cpu().numpy(), Ir) and np.array_equal(D.cpu().numpy(), Dr)


def test_simulated_shards_nan_and_infinite_distances():
    """NaN rows of several bit patterns and +-inf rows across every cut: the merge ranks NaN after +inf, by id, as the
    single index does, and both return the NaN 0x7FFFFFFF."""
    g = torch.Generator(device="cuda").manual_seed(7)
    X = torch.randn((150, 128), generator=g, device="cuda")        # 30 NaN rows: every top-128 reaches them
    nans = torch.tensor([0x7FC00000, 0xFFC00000, 0x7FC0BEEF, 0xFFFFFFFF], dtype=torch.int64).to(torch.int32)
    X[3::5, 0] = nans.view(torch.float32).cuda().repeat(8)[:30]
    X[[1, 75, 149], 1] = float("inf")
    X[[2, 76], 2] = -float("inf")
    Q = torch.randn((6, 128), generator=g, device="cuda")
    Q[5, 0] = float("nan")
    D, I = _check_shards(X, Q, 128)
    bits = D.cpu().numpy().view(np.uint32)
    assert np.all(bits[np.isnan(D.cpu().numpy())] == 0x7FFFFFFF) and np.isnan(D[0, -1].item())
    assert torch.equal(I[5], torch.arange(128, device="cuda"))      # a NaN query: every distance NaN, id order


# ---------------------------------------------------------------------------------------------- NCCL, one process per GPU
N_FILE, D_FILE, B_FILE = 50_003, 768, 16
N_SYN, D_SYN = synth.EMB_BLOCK + 4097, 64


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        res = {}
        Q = np.load(os.path.join(out_dir, "q.npy"))
        for name in ("big", "small"):
            ix = read_index(os.path.join(out_dir, f"{name}.index"), device=dev, sharded=True)
            lo, hi = sharding.shard_range(ix.ntotal, rank, world)
            assert isinstance(ix, ShardedIndexFlatL2) and ix.shard.ntotal == hi - lo and ix.row_base == lo
            for k in (5, 128):
                Dn, In = ix.search(Q, k)
                Dt, It = ix.search(torch.from_numpy(Q).to(dev), k)
                assert isinstance(Dn, np.ndarray) and Dt.device == dev
                assert np.array_equal(Dt.cpu().numpy(), Dn) and np.array_equal(It.cpu().numpy(), In)
                res[f"{name}_D{k}"], res[f"{name}_I{k}"] = Dn, In
            assert ix.last_stats()["launches"] >= 2
        # every rank builds only its own synthetic rows, and the same query batch from the shape alone
        lo, hi = sharding.shard_range(N_SYN, rank, world)
        shard = IndexFlatL2(D_SYN, dev)
        shard.add(synth.dense_rows(N_SYN, D_SYN, device=dev, row_lo=lo, row_hi=hi))
        full = synth.dense_rows(N_SYN, D_SYN, device=dev)
        assert torch.equal(shard.rows(), full[lo:hi])
        q = synth.dense_queries_of(N_SYN, D_SYN, 33, device=dev)
        assert torch.equal(q, synth.dense_queries(full, 33))
        del full
        D, I = ShardedIndexFlatL2(shard, lo).search(q, 10)
        res["syn_D"], res["syn_I"] = D.cpu().numpy(), I.cpu().numpy()
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("world", [2, 4])
def test_nccl_row_shards_equal_single_index_and_oracle(tmp_path, world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, this box has {torch.cuda.device_count()}")
    import torch.multiprocessing as mp
    rows = synth.dense_rows(N_FILE, D_FILE)
    Q = synth.dense_queries(rows, B_FILE)
    single = IndexFlatL2(D_FILE)
    single.add(rows)
    write_index(single, str(tmp_path / "big.index"))
    tiny = IndexFlatL2(D_FILE)
    tiny.add(rows[:world - 1])                               # more ranks than rows: the last rank holds none
    write_index(tiny, str(tmp_path / "small.index"))
    np.save(tmp_path / "q.npy", Q.cpu().numpy())
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for name, ix in (("big", single), ("small", tiny)):
        for k in (5, 128):
            Ds, Is = ix.search(Q, k)
            Dr, Ir = fo.search_canonical_torch(Q, ix.rows(), k)
            assert np.array_equal(Is.cpu().numpy(), Ir) and np.array_equal(Ds.cpu().numpy(), Dr)
            for r in range(world):
                got = np.load(tmp_path / f"r{r}.npz")
                assert np.array_equal(got[f"{name}_I{k}"], Ir), f"rank {r} {name} k={k}: ids differ"
                assert np.array_equal(got[f"{name}_D{k}"], Dr), f"rank {r} {name} k={k}: distances differ"
    syn = IndexFlatL2(D_SYN)
    syn.add(synth.dense_rows(N_SYN, D_SYN))
    Ds, Is = syn.search(synth.dense_queries(syn.rows(), 33), 10)
    for r in range(world):
        got = np.load(tmp_path / f"r{r}.npz")
        assert np.array_equal(got["syn_I"], Is.cpu().numpy()) and np.array_equal(got["syn_D"], Ds.cpu().numpy())
