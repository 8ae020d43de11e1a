"""probing_rag_b200 -- the B200-native retrieval hot path of Probing-RAG.

Batched BM25 scoring + top-k over a CSR inverted index in HBM, the per-shard list merge and
the prober gate, exact dense (faiss IndexFlatL2 / IndexFlatIP) search, as hand-written sm_100a CUDA behind a C ABI (include/probing_rag.h), with a
Python host side that mirrors the reference's retriever / prober interfaces
(/root/reference/exp_rag.py:236-242, 381-415, 426-428; utils.py:29-57, 282-330).
"""
from .dense import (METRIC_INNER_PRODUCT, METRIC_L2, IndexFlatIP, IndexFlatL2,   # noqa: F401
                    ShardedIndexFlatIP, ShardedIndexFlatL2, read_index, write_index)
from .index import BM25Index, merge_topk                       # noqa: F401
from .retriever import (BM25Retriever, Document, NodeWithScore,   # noqa: F401
                        SimpleDocumentStore, TextNode)

__version__ = "0.1.0"
