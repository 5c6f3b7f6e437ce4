"""Import the reference's OWN hot-path modules unmodified (TEST INFRASTRUCTURE, fixture generation only).

The reference tree is not part of this repository: ``SENTIO_REFERENCE_ROOT`` points at a checkout of chernistry/sentio.
This loader is used ONLY by tests/golden/make_golden.py to produce the committed fixtures; the tests themselves read the
fixtures and never the reference.  Packages that cannot be installed offline are stubbed in sys.modules (SURVEY.md
Appendix D): rank_bm25 -> oracle/rank_bm25_port.py, qdrant_client -> a NumPy exact-cosine stand-in, langchain /
langgraph -> empty shells.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("SENTIO_REFERENCE_ROOT", "")


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "src", "core", "retrievers"))


class _Any:
    def __init__(self, *a, **k):
        pass


class ScoredPoint:
    def __init__(self, id, score, payload):
        self.id, self.score, self.payload = id, score, payload


class NumpyQdrantClient:
    """Exact-cosine stand-in for QdrantClient (search / scroll / collection_exists)."""

    def __init__(self):
        self.collections = {}

    def add_collection(self, name, rows16, ids, payloads):
        self.collections[name] = (np.asarray(rows16), list(ids), list(payloads))

    def collection_exists(self, collection_name):
        return collection_name in self.collections

    def search(self, collection_name, query_vector, limit=10, with_payload=True, with_vectors=False, **kw):
        from . import dense as dense_oracle

        rows16, ids, payloads = self.collections[collection_name]
        idx, sc = dense_oracle.dense_topk(rows16, np.asarray(query_vector, dtype=np.float32), limit)
        return [ScoredPoint(ids[i], float(s), payloads[i]) for i, s in zip(idx, sc)]

    def scroll(self, collection_name, limit=100, offset=None, with_payload=True, with_vectors=False, **kw):
        rows16, ids, payloads = self.collections[collection_name]
        start = int(offset or 0)
        stop = min(len(ids), start + limit)
        pts = [ScoredPoint(ids[i], 0.0, payloads[i]) for i in range(start, stop)]
        return pts, (stop if stop < len(ids) else None)


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


_loaded = None


def load():
    """Returns a namespace with the reference classes; installs the stubs on first use."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT!r}: set SENTIO_REFERENCE_ROOT")
    from . import rank_bm25_port

    if "rank_bm25" not in sys.modules:
        _stub("rank_bm25", BM25Okapi=rank_bm25_port.BM25Okapi, BM25Plus=rank_bm25_port.BM25Plus)
    if "qdrant_client" not in sys.modules:
        _stub("qdrant_client", QdrantClient=NumpyQdrantClient, AsyncQdrantClient=_Any)
        _stub("qdrant_client.http", models=types.SimpleNamespace())
        _stub("qdrant_client.http.models")
    for name, attrs in [("langchain_core", {}), ("langchain_core.documents", {"Document": _Any}),
                        ("langchain_core.embeddings", {"Embeddings": _Any}),
                        ("langchain_core.vectorstores", {"VectorStore": object}),
                        ("langchain_core.language_models", {"BaseChatModel": _Any}),
                        ("langchain_core.prompts", {"ChatPromptTemplate": _Any}),
                        ("langgraph", {}), ("langgraph.graph", {"END": "__end__", "StateGraph": _Any}),
                        ("langchain_text_splitters", {"CharacterTextSplitter": _Any,
                                                      "RecursiveCharacterTextSplitter": _Any})]:
        if name not in sys.modules:
            _stub(name, **attrs)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import logging

    logging.getLogger("src").setLevel(logging.ERROR)
    from src.core.models.document import Document
    from src.core.retrievers.dense import DenseRetriever
    from src.core.retrievers.hybrid import HybridRetriever
    from src.core.retrievers.scorers import KeywordMatchScorer, MMRScorer, SemanticSimilarityScorer
    from src.core.retrievers.sparse import BM25Retriever

    ns = types.SimpleNamespace(Document=Document, DenseRetriever=DenseRetriever, HybridRetriever=HybridRetriever,
                               BM25Retriever=BM25Retriever, KeywordMatchScorer=KeywordMatchScorer, MMRScorer=MMRScorer,
                               SemanticSimilarityScorer=SemanticSimilarityScorer, NumpyQdrantClient=NumpyQdrantClient)
    try:
        from src.core.graph.nodes import create_reranker_node, create_retriever_node
        from src.core.graph.state import create_initial_state

        ns.create_retriever_node = create_retriever_node
        ns.create_reranker_node = create_reranker_node
        ns.create_initial_state = create_initial_state
    except Exception as exc:  # pragma: no cover - graph import is optional for the fixtures
        ns.graph_import_error = exc
    _loaded = ns
    return ns
