"""The reference's OWN LangGraph node functions (src/core/graph/nodes.py:37-227) drive this repository's retriever /
reranker classes -- north_star's acceptance sentence ("so the LangGraph nodes ... call it unchanged") as a test.

tests/golden/reference_nodes.json holds what the unmodified reference nodes returned when they drove HybridRetriever and
B200Reranker on the oracle-backed engine double (tests/golden/make_golden.py), together with the inputs.  The nodes call
``retriever.retrieve(query, top_k=...)`` / ``reranker.rerank(query=, docs=, top_k=)`` and copy what comes back, so the
classes called the same way must return the recorded documents:

* CPU (`not gpu`): the classes on the oracle-backed engine double (host logic).
* GPU: the same classes on the real engine / C ABI.
"""
import threading

import numpy as np
import pytest

from conftest import load_golden
from helpers import HashEmbedder
from sentio_b200.cross_encoder import CrossEncoderWeights
from sentio_b200.document import Document
from sentio_b200.rerankers.b200_reranker import B200Reranker
from sentio_b200.retrievers.dense import DenseRetriever
from sentio_b200.retrievers.hybrid import HybridRetriever

GOLD = load_golden("reference_nodes")
DIM = GOLD["dim"]
TEXTS = GOLD["texts"]
IDS = GOLD["ids"]


def _build(make_store, make_sparse, engine):
    emb = HashEmbedder(DIM)
    vecs = np.asarray(emb.embed_many_sync(TEXTS), dtype=np.float32)
    store = make_store(vecs, IDS, GOLD["payloads"])
    corpus = [Document(id=i, text=t, metadata={"source": "corpus"}) for i, t in zip(IDS, TEXTS)]
    dense = DenseRetriever(client=store, embedder=emb, collection_name="Sentio_docs")
    hr = HybridRetriever(dense_retriever=dense, sparse_retriever=make_sparse(corpus), rrf_k=60, scorer_plugins=[],
                         fusion_method="rrf", engine=engine)
    rr = B200Reranker(weights=CrossEncoderWeights.random(GOLD["ce_config"], seed=GOLD["ce_seed"]), engine=engine,
                      seq_len=GOLD["seq_len"])
    return hr, rr


def _same_metadata(got, want):
    """Rank-fusion scores bit-exact, raw cosines to fp64 summation order, everything else equal."""
    assert got.keys() == want.keys(), (got, want)
    for key, w in want.items():
        if isinstance(w, float) and key not in ("score", "hybrid_score"):
            assert np.isclose(got[key], w, rtol=1e-9, atol=1e-12), (key, got[key], w)
        else:
            assert got[key] == w, (key, got[key], w)


def _check_rerank(rr, case, out, exact):
    """``out`` = B200Reranker.rerank on the node's prepared copies vs the node's recorded output.  On the oracle engine
    the order is the recorded one; on the GPU the cross-encoder runs in fp16 / fp32 (rel 1e-3, abs 1e-4 vs the oracle)
    and this random-init model scores all candidates within ~1e-4 of each other, so ranks may swap inside that band."""
    want = case["reranked"]
    assert len(out) == len(want) == min(GOLD["rerank_top_k"], len(case["retrieved"]))
    assert all(set(d.metadata) == set(w[2]) for d, w in zip(out, want))
    sc = [d.metadata["rerank_score"] for d in out]
    assert sc == sorted(sc, reverse=True)
    assert all(0.0 <= d.metadata["score"] <= 1.0 and d.metadata["score"] == d.metadata["rerank_score"] for d in out)
    if exact:
        assert [d.id for d in out] == [w[0] for w in want]
        assert [d.text for d in out] == [w[1] for w in want]
        assert np.allclose(sc, [w[2]["rerank_score"] for w in want], rtol=1e-6, atol=0)
        return
    rtol, atol = 1e-3, 1e-4
    texts = [t for _, t, _ in case["retrieved"]]
    every = dict(zip([i for i, _, _ in case["retrieved"]], map(float, rr.score_pairs(case["query"], texts))))
    for doc_id, _, meta in want:                               # the recorded top documents score the same here
        assert np.isclose(every[doc_id], meta["rerank_score"], rtol=rtol, atol=atol), (doc_id, every[doc_id], meta)
    assert all(d.metadata["rerank_score"] == every[d.id] for d in out)
    floor = min(meta["rerank_score"] for _, _, meta in want)
    for d in out:                                              # anything else got in through a near tie at the cut
        assert d.id in {w[0] for w in want} or every[d.id] >= floor - 2 * (atol + rtol * floor), (d.id, every[d.id])
    assert np.allclose(sc, [w[2]["rerank_score"] for w in want], rtol=rtol, atol=atol)


def _drive_like_the_nodes(hr, rr, exact_rerank):
    for case in GOLD["cases"]:
        q = case["query"]
        # ---- retrieve_node == HybridRetriever.retrieve (nodes.py:51-119)
        got = hr.retrieve(q, top_k=GOLD["retrieve_top_k"])
        want = case["retrieved"]
        assert [d.id for d in got] == [w[0] for w in want], q
        assert [d.text for d in got] == [w[1] for w in want] and all(d.text for d in got)
        for d, w in zip(got, want):
            _same_metadata(d.metadata, w[2])
        assert case["retrieve_metadata"] == {"retriever_type": type(hr).__name__, "retrieved_count": len(got)}
        # ---- metadata.user_top_k overrides the node's top_k (nodes.py:64-69)
        want5 = case["retrieved_user_top_k_5"]  # (a hybrid top-5 is not a prefix of the top-10: the sub-retrievers get top_k too)
        assert [d.id for d in hr.retrieve(q, top_k=5)] == want5 and len(want5) <= 5
        # ---- rerank_node == B200Reranker.rerank on the node's prepared copies (nodes.py:138-227)
        if not want:
            assert case["reranked"] == []
            continue
        prepared = [Document(id=i, text=t, metadata=dict(m)) for i, t, m in want]
        out = rr.rerank(query=q, docs=prepared, top_k=GOLD["rerank_top_k"])
        _check_rerank(rr, case, out, exact_rerank)
        assert case["rerank_metadata"] == {**case["retrieve_metadata"], "reranker_type": type(rr).__name__,
                                           "reranked_count": len(out)}

    # ---- a raising retriever lands in metadata["retriever_error"], the graph continues without documents: the
    # HybridRetriever propagates a dense failure with its message, which is what the node records
    boom = GOLD["raising_retriever"]
    assert boom["metadata"] == {"retriever_error": boom["error"]} and boom["retrieved"] == []

    class Boom:
        def retrieve(self, query, top_k=10):
            raise RuntimeError(boom["error"])

    failing = HybridRetriever(dense_retriever=Boom(), sparse_retriever=hr._sparse_retriever, rrf_k=60,
                              scorer_plugins=[], fusion_method="rrf", engine=hr._engine)
    with pytest.raises(RuntimeError) as exc:
        failing.retrieve("q", top_k=3)
    assert str(exc.value) == boom["error"]
    # ---- no documents: rerank_node returns the state untouched; the reranker itself returns [] for no documents
    assert GOLD["no_documents"] == {"metadata": {}, "reranked": []}
    assert rr.rerank(query="q", docs=[], top_k=GOLD["rerank_top_k"]) == []


def test_reference_nodes_drive_the_repo_classes_host_logic(monkeypatch):
    from oracle_engine import OracleEngine
    from sentio_b200.retrievers import sparse as sparse_mod
    from test_hybrid_e2e import _OracleStore

    monkeypatch.delenv("BM25_VARIANT", raising=False)
    monkeypatch.setattr(sparse_mod, "B200Engine", lambda device=0: OracleEngine())
    eng = OracleEngine()
    hr, rr = _build(_OracleStore, lambda corpus: sparse_mod.BM25Retriever(documents=corpus), eng)
    _drive_like_the_nodes(hr, rr, exact_rerank=True)


@pytest.mark.gpu
def test_reference_nodes_drive_the_repo_classes_on_the_gpu(engine, monkeypatch):
    from sentio_b200.retrievers.sparse import BM25Retriever
    from sentio_b200.vector_store import B200VectorStore

    monkeypatch.delenv("BM25_VARIANT", raising=False)

    def make_store(vecs, ids, payloads):
        st = B200VectorStore(0)
        st.create_collection("Sentio_docs", vecs, ids=ids, payloads=payloads)
        return st

    hr, rr = _build(make_store, lambda corpus: BM25Retriever(documents=corpus), engine)
    _drive_like_the_nodes(hr, rr, exact_rerank=False)


@pytest.mark.gpu
def test_concurrent_retrieve_async_on_one_context(engine, monkeypatch):
    """retrievers/base.py:37-42 dispatches ``retrieve`` to the default thread pool, so one engine context is entered
    from several Python threads at once (ctypes releases the GIL): every call must return exactly the serial answer."""
    import asyncio

    from sentio_b200.retrievers.sparse import BM25Retriever
    from sentio_b200.vector_store import B200VectorStore

    monkeypatch.delenv("BM25_VARIANT", raising=False)

    def make_store(vecs, ids, payloads):
        st = B200VectorStore(0)
        st.create_collection("Sentio_docs", vecs, ids=ids, payloads=payloads)
        return st

    hr, rr = _build(make_store, lambda corpus: BM25Retriever(documents=corpus), engine)
    queries = [f"topic{i % 9} w{i % 13} alpha{i % 5}" for i in range(48)]
    # ids only: like the reference, BM25Retriever hands out the SHARED corpus Documents and the fusion writes
    # metadata["hybrid_score"] into them in place (sparse.py:189-197, hybrid.py:296-297), so under concurrency a document's
    # score field belongs to whichever query wrote last -- the ranking of each call is what must be stable
    serial = [[d.id for d in hr.retrieve(q, top_k=10)] for q in queries]

    async def one(q):
        docs = await hr.retrieve_async(q, top_k=10)
        return [d.id for d in docs]

    async def hammer():
        return await asyncio.gather(*[one(q) for q in queries])

    assert asyncio.run(hammer()) == serial
    # raw threads on the engine itself: dense / BM25 / rerank entry points interleaved on ONE sb_ctx
    emb = HashEmbedder(DIM)
    qv = np.asarray(emb.embed_many_sync(queries), dtype=np.float32)
    st = hr._dense._client  # the B200VectorStore behind the dense retriever
    want = [st.search("Sentio_docs", list(v), limit=7) for v in qv]
    errors, got = [], [None] * len(queries)

    def worker(lo, hi):
        try:
            for i in range(lo, hi):
                got[i] = st.search("Sentio_docs", list(qv[i]), limit=7)
                rr.score_pairs(queries[i], TEXTS[i:i + 3])
        except Exception as exc:  # pragma: no cover
            errors.append(exc)

    threads = [threading.Thread(target=worker, args=(j * 12, (j + 1) * 12)) for j in range(4)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
    assert [[(p.id, p.score) for p in r] for r in got] == [[(p.id, p.score) for p in r] for r in want]
