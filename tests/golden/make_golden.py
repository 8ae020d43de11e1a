"""Generate tests/golden/*.npz.  Run in the BUILD container only (needs /root/reference):

    python tests/golden/make_golden.py

prober_golden.npz  outputs of the REFERENCE's own `ImprovedProbe` (AST-extracted from
                   /root/reference/utils.py:29-57, unmodified) on seeded inputs/weights that
                   oracle/prober_oracle.py regenerates anywhere; digests guard RNG drift.
bm25_golden.npz    a small corpus scored by the oracle's literal per-document builder
                   (oracle/bm25_oracle.build_index_loop).  The real bm25s/llama-index
                   packages are absent (SURVEY 8c), so this fixture pins the oracle against
                   regressions, not against the library: BM25 parity stays "unpinned".
"""
import ast
import hashlib
import os
import sys

import numpy as np
import torch
from torch import nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import bm25_oracle as bo          # noqa: E402
from oracle import prober_oracle as po        # noqa: E402

REF_UTILS = "/root/reference/utils.py"


def load_reference_improved_probe():
    src = open(REF_UTILS).read()
    tree = ast.parse(src)
    node = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "ImprovedProbe")
    mod = ast.Module(body=[node], type_ignores=[])
    ns = {"nn": nn, "torch": torch}
    exec(compile(mod, REF_UTILS, "exec"), ns)
    return ns["ImprovedProbe"], (node.lineno, node.end_lineno)


def make_prober_golden():
    RefProbe, lines = load_reference_improved_probe()
    n = 48
    x = po.make_hidden_states(n, seed=0)
    ref_probers, ora_probers, digests = [], [], []
    for layer in po.PROBE_LAYERS:
        sd = po.make_prober_state(layer)
        rp = RefProbe(input_size=po.D_MODEL, output_size=po.N_CLASSES)
        rp.load_state_dict(sd)
        rp.eval()
        op = po.OracleImprovedProbe(po.D_MODEL, po.N_CLASSES)
        op.load_state_dict(sd)
        op.eval()
        assert list(rp.state_dict().keys()) == list(op.state_dict().keys())
        assert sum(p.numel() for p in rp.parameters()) == 1318914     # exp_parameter_check.py:52
        ref_probers.append(rp)
        ora_probers.append(op)
        digests.append(po.state_digest(sd))
    ref_logits = po.prober_logits(ref_probers, x)
    ora_logits = po.prober_logits(ora_probers, x)
    assert torch.equal(ref_logits, ora_logits), "oracle restatement differs from the reference class"
    # the gate exactly as exp_rag.py:407-415 writes it, per row
    softmax_f = torch.nn.Softmax(dim=1)
    psum = torch.zeros(n, 2)
    retrieve = np.zeros((3, n), dtype=np.bool_)
    thetas = np.array([0.0, -1.0, 1.0], dtype=np.float32)
    for i in range(n):
        logits = [ref_logits[i:i + 1, p] for p in range(6)]
        acc = torch.zeros_like(logits[0].squeeze())
        for num in range(0, len(logits)):
            acc += (softmax_f(logits[num])).squeeze()
        psum[i] = acc
        for j, th in enumerate(thetas):
            retrieve[j, i] = not (acc[0].item() + float(th) < acc[1].item())
    o_psum, o_ret = po.gate(ref_logits, 0.0, 0)
    assert torch.allclose(o_psum, psum, atol=1e-6) and np.array_equal(o_ret.numpy(), retrieve[0])
    np.savez_compressed(
        os.path.join(HERE, "prober_golden.npz"),
        logits=ref_logits.numpy(), probsum=psum.numpy(), retrieve=retrieve, thetas=thetas,
        state_digests=np.array(digests), x_digest=hashlib.sha256(x.numpy().tobytes()).hexdigest(),
        n=n, ref_lines=np.array(lines), torch_version=torch.__version__)
    print("prober_golden.npz: logits", tuple(ref_logits.shape), "retrieve rate",
          retrieve.mean(axis=1))


def make_bm25_golden():
    rng = np.random.default_rng(99)
    n_docs, vocab = 300, 64
    docs = []
    for i in range(n_docs):
        ln = int(rng.integers(3, 40))
        docs.append(np.minimum(rng.zipf(1.4, size=ln) - 1, vocab - 1).astype(np.int32))
    docs[7] = docs[3].copy()                       # exact duplicate docs -> exact score ties
    docs[250] = docs[3].copy()
    idx = bo.build_index_loop(docs, vocab)
    queries = [np.array(q, dtype=np.int32) for q in
               ([0], [1, 0], [5, 5, 2], [63], [10, 3, 0, 1, 2, 7], [], [40, 41, 42], [2, 0, 2, 0, 2])]
    q_indptr = np.zeros(len(queries) + 1, dtype=np.int64)
    q_indptr[1:] = np.cumsum([len(q) for q in queries])
    q_terms = np.concatenate(queries).astype(np.int32)
    k = 10
    scores, ids = bo.retrieve_batch(idx, q_indptr, q_terms, k)
    np.savez_compressed(
        os.path.join(HERE, "bm25_golden.npz"),
        tokens=np.concatenate(docs).astype(np.int32),
        doc_lens=np.array([len(d) for d in docs], dtype=np.int32), vocab=vocab,
        data=idx["data"], indices=idx["indices"], indptr=idx["indptr"],
        q_indptr=q_indptr, q_terms=q_terms, k=k, scores=scores, ids=ids)
    print("bm25_golden.npz: nnz", len(idx["data"]), "queries", len(queries))


if __name__ == "__main__":
    torch.manual_seed(0)
    torch.set_num_threads(8)        # test_prober_oracle.GOLDEN_THREADS: the float32 logits depend on the thread count
    make_prober_golden()
    make_bm25_golden()
