"""Exact search over fp16 rows at the size bench_dense.py measures -- 21,015,324 x 768 -- against the batched reference
(tests/flat_fast_oracle.py) over the fp16-decoded rows, ids and distance or score bits, for both metrics.  Needs a
B200.  PR_SKIP_FULL=1 skips the file.

One full-size index is on the device at a time: the resident index of test_gpu_flat_fullsize (shared with the full-size
range tests, 97 GB) is freed first.  The fp16 index is built by add() from row blocks generated one at a time, so no
f32 copy of the whole matrix exists, and the reference decodes the codes one chunk of rows at a time: the top-128 of
each chunk (exact values do not depend on the chunk), merged in the canonical order (value key, row id)."""
import gc
import os
import time

import numpy as np
import pytest
import torch

import flat_fast_oracle as ffo
from oracle import flat_ip_oracle as fio
from probing_rag_b200 import METRIC_INNER_PRODUCT, METRIC_L2, IndexScalarQuantizer, ScalarQuantizer, synth

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(os.environ.get("PR_SKIP_FULL") == "1", reason="PR_SKIP_FULL=1")]

N_ROWS, D = synth.N_DOCS_WIKI, 768
NQ, N_SAMPLE, K_MAX = 512, 128, 128
ADD_ROWS = 1 << 22          # rows generated and added per add() call
REF_ROWS = 1 << 21          # decoded rows per reference chunk (6.4 GB of f32)


def _bits(x):
    return np.ascontiguousarray(x.cpu().numpy() if isinstance(x, torch.Tensor) else x).view(np.uint32)


def _free():
    gc.collect()
    torch.cuda.empty_cache()


def _reference(index, Q, metric):
    """The top-K_MAX of every query over the decoded rows, chunk by chunk, merged canonically."""
    Ds, Is = [], []
    codes = index.codes()
    for a in range(0, codes.shape[0], REF_ROWS):
        Xc = codes[a:a + REF_ROWS].float()
        Dc, Ic = ffo.search_fast(Q, Xc, K_MAX, metric)
        del Xc
        Ds.append(Dc)
        Is.append(Ic + a)
    Dall, Iall = np.concatenate(Ds, axis=1), np.concatenate(Is, axis=1)
    key = Dall.view(np.uint32) if metric == "l2" else fio.ip_key(Dall)   # finite values: the refine's key order
    out_D, out_I = np.empty((Q.shape[0], K_MAX), np.float32), np.empty((Q.shape[0], K_MAX), np.int64)
    for b in range(Q.shape[0]):
        o = np.lexsort((Iall[b], key[b]))[:K_MAX]
        out_D[b], out_I[b] = Dall[b, o], Iall[b, o]
    return out_D, out_I


@pytest.mark.parametrize("metric", ["l2", "ip"])
def test_sampled_batch_against_the_fast_reference(metric):
    import test_gpu_flat_fullsize as fs
    fs._free()
    _free()
    print(f"[sq fullsize] {metric}: {torch.cuda.memory_allocated() / 2 ** 30:.1f} GiB allocated before the build",
          flush=True)
    t0 = time.perf_counter()
    index = IndexScalarQuantizer(D, ScalarQuantizer.QT_fp16, METRIC_L2 if metric == "l2" else METRIC_INNER_PRODUCT)
    for a in range(0, N_ROWS, ADD_ROWS):
        index.add(synth.dense_rows(N_ROWS, D, row_lo=a, row_hi=min(N_ROWS, a + ADD_ROWS)))
        _free()
    assert index.ntotal == N_ROWS
    Q = synth.dense_queries_of(N_ROWS, D, NQ)
    sel = np.sort(np.random.default_rng(7).choice(NQ, N_SAMPLE, replace=False))
    ref_D, ref_I = _reference(index, Q[torch.from_numpy(sel).cuda()].contiguous(), metric)
    _free()
    print(f"[sq fullsize] {metric}: index and reference in {time.perf_counter() - t0:.1f} s", flush=True)
    for k in (10, K_MAX):
        D_, I_ = index.search(Q, k)
        assert np.array_equal(I_.cpu().numpy()[sel], ref_I[:, :k]), f"{metric} k={k}: ids differ"
        assert np.array_equal(_bits(D_)[sel], _bits(ref_D[:, :k])), f"{metric} k={k}: value bits differ"
        st = index.last_stats()
        print(f"[sq fullsize] {metric} k={k}: candidates {st['candidates']:,}, fallbacks {st['fallback_queries']}",
              flush=True)
    del index
    _free()
