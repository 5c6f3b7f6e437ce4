"""CPU-only coverage of host logic added around the hot path: Pyserini strategy fallback (factory.py:150-176 of the
reference), the embedder's tokeniser / BaseEmbedder surface with a fake engine, the selector device-input helper."""
import asyncio

import numpy as np
import pytest

from sentio_b200.document import Document


class _FakeEmbedder:
    def embed_sync(self, text):
        return [1.0, 0.0]

    def embed_many_sync(self, texts):
        return [[1.0, 0.0] for _ in texts]


class _FakeClient:
    def collection_exists(self, collection_name):
        return False

    def scroll(self, **kw):
        return [], None


def test_pyserini_strategy_falls_back_like_the_reference(monkeypatch, tmp_path):
    from sentio_b200.retrievers import factory, get_retriever
    from sentio_b200.retrievers import sparse as sparse_mod

    built = []

    class _Stub(sparse_mod.BM25Retriever):
        def __init__(self, documents=None, variant="okapi", **kw):
            built.append((len(documents or []), variant))

    monkeypatch.setattr(factory, "BM25Retriever", _Stub)
    monkeypatch.setenv("RETRIEVAL_STRATEGY", "pyserini")
    monkeypatch.setenv("BM25_INDEX_DIR", str(tmp_path / "missing"))
    docs = [Document(id="a", text="x y"), Document(id="b", text="y z")]
    r = factory.create_retriever_from_env(_FakeClient(), _FakeEmbedder(), corpus_docs=docs)
    assert isinstance(r, _Stub) and built == [(2, "okapi")]  # RuntimeError inside -> in-memory BM25 (factory.py:158-163)
    with pytest.raises(RuntimeError):                        # get_retriever("pyserini") raises like the reference class
        get_retriever("pyserini", index_dir=str(tmp_path / "missing"))
    (tmp_path / "idx").mkdir()
    with pytest.raises(RuntimeError):                        # an index directory alone is not enough: no JVM / Lucene reader
        get_retriever("lucene", index_dir=str(tmp_path / "idx"))
    with pytest.raises(ValueError):
        get_retriever("nope")


def test_embedding_tokeniser_frames_and_truncates():
    from sentio_b200.embedder import tokenize_for_embedding
    from sentio_b200.index import CLS_ID, PAD_ID, SEP_ID, _hash_token

    ids, tt, lens = tokenize_for_embedding(["Hello  World", "", "w " * 500], seq_len=16)
    assert list(ids[0, :4]) == [CLS_ID, _hash_token("hello"), _hash_token("world"), SEP_ID] and lens[0] == 4
    assert np.all(ids[0, 4:] == PAD_ID) and np.all(tt == 0)
    assert list(ids[1, :2]) == [CLS_ID, SEP_ID] and lens[1] == 2
    assert lens[2] == 16 and ids[2, 0] == CLS_ID and ids[2, 15] == SEP_ID


def test_embedder_surface_with_fake_engine():
    from sentio_b200.cross_encoder import CrossEncoderWeights
    from sentio_b200.embedder import B200Embedder

    calls = []

    class _Eng:
        def enc_load(self, blob, cfg, pw, pb):
            self.dim = pw.shape[0] if pw is not None else cfg["hidden"]

        def enc_dim(self):
            return self.dim

        def enc_embed(self, ids, tt, lens, normalize=True):
            calls.append(ids.shape[0])
            v = np.zeros((ids.shape[0], self.dim), np.float32)
            v[:, 0] = lens
            return v

    cfg = dict(vocab_size=30522, hidden=128, layers=1, heads=4, intermediate=128, max_pos=64, type_vocab=2, ln_eps=1e-12)
    emb = B200Embedder(weights=CrossEncoderWeights.random(cfg, seed=1), dimension=256, seq_len=32, engine=_Eng())
    assert emb.dimension == 256
    out = emb.embed_many_sync(["a b", "c", "a b"])
    assert [v[0] for v in out] == [4.0, 3.0, 4.0] and calls == [3]
    assert emb.embed_sync("a b")[0] == 4.0 and calls == [3]          # served from the cache
    assert emb.stats["cache_hits"] == 1 and emb.stats["total_requests"] == 4
    assert asyncio.run(emb.embed_async_many(["zz top"]))[0][0] == 4.0 and calls == [3, 1]
    assert asyncio.run(emb.warm_up()) is True
    asyncio.run(emb.close())
    emb.reset_stats()
    assert emb.stats["total_requests"] == 0


def test_selector_chars_matches_the_text_the_selector_uses():
    from sentio_b200.selector import selector_chars

    assert selector_chars(Document(id="1", text="abcd")) == 4
    assert selector_chars(Document(id="2", text="", metadata={"content": "xyz"})) == 3
    assert selector_chars(Document(id="3", text="   ")) == 0
    assert selector_chars(Document(id="4", text="", metadata={})) == 0


def test_multi_gpu_layout_planner():
    from sentio_b200.pipeline import plan_layout

    assert plan_layout(1, 2.05) == (1, 1)
    assert plan_layout(8, 2.05, "auto") == (1, 8)              # the metric's corpus fits one GPU: replicate
    assert plan_layout(8, 2.05, "corpus") == (8, 1)            # north_star's layout
    assert plan_layout(8, 2.05, "queries") == (1, 8)
    assert plan_layout(8, 200.0, "auto", budget_gb=64.0) == (4, 2)   # partition only as much as capacity requires
    assert plan_layout(8, 2000.0, "auto", budget_gb=64.0) == (8, 1)  # never more shards than GPUs
    assert plan_layout(4, 2.05, "auto", corpus_shards=2) == (2, 2)
    with pytest.raises(ValueError):
        plan_layout(8, 2.05, corpus_shards=3)
    with pytest.raises(ValueError):
        plan_layout(8, 2.05, "banana")


def test_reranker_batch_equals_per_query_with_fake_engine():
    """B200Reranker.rerank_batch (one forward over all pairs) == rerank per job; blank / empty jobs degrade per job."""
    from sentio_b200.cross_encoder import CrossEncoderWeights
    from sentio_b200.rerankers.b200_reranker import B200Reranker
    from sentio_b200.rerankers.base import RerankingResult

    class _Eng:
        device = 0

        def ce_load(self, blob, cfg):
            pass

        def ce_score(self, ids, tt, lens):  # deterministic pseudo relevance from the token ids
            s = (ids.astype(np.int64).sum(axis=1) % 97) / 97.0
            return s, s.astype(np.float32)

    cfg = dict(vocab_size=30522, hidden=128, layers=1, heads=4, intermediate=128, max_pos=64, type_vocab=2, ln_eps=1e-12)
    mk = lambda: [[Document(id=f"a{i}", text=f"w{i} w{i + 3}") for i in range(7)],
                  [Document(id="b0", text="", metadata={"content": "w5 w6"}), Document(id="b1", text="w9")], [],
                  [Document(id=f"c{i}", text=f"w{2 * i}", metadata={"score": 0.5}) for i in range(4)]]
    qs = ["w1 w2", "w5", "w7", "   "]
    rr = B200Reranker(weights=CrossEncoderWeights.random(cfg, seed=1), engine=_Eng(), seq_len=32)
    a = rr.rerank_batch(qs, mk(), top_k=3)
    b = [rr.rerank(q, d, top_k=3) for q, d in zip(qs, mk())]
    assert [[(d.id, d.metadata.get("rerank_score"), d.text) for d in x] for x in a] == \
           [[(d.id, d.metadata.get("rerank_score"), d.text) for d in x] for x in b]
    assert a[2] == [] and [d.metadata["rerank_score"] for d in a[3]] == [1.0, 0.9, 0.8]
    res = RerankingResult(a[0], None, None)
    assert len(res) == 3 and res.top_document is a[0][0] and list(res) == a[0] and res.metadata == {}


def test_every_module_imports_without_a_gpu():
    """Importing the package (all modules) must not touch CUDA or need the built library."""
    import importlib
    import pkgutil

    import sentio_b200

    names = [m.name for m in pkgutil.walk_packages(sentio_b200.__path__, "sentio_b200.")]
    assert {"sentio_b200.embedder", "sentio_b200.selector", "sentio_b200.pipeline"} <= set(names)
    for name in names:
        if name.endswith(".build") or "libsentio_b200" in name:  # the C-ABI library is not a Python extension module
            continue
        importlib.import_module(name)


def test_bm25_persistence_large_top_k_and_scroll_corpus_host_logic(tmp_path, monkeypatch):
    """Host logic of sparse.py:102-157 (save / load into a fresh object), of top_k beyond one kernel call and of the
    factory's Qdrant-payload scroll (factory.py:83-133), on the oracle-backed engine double."""
    import pickle

    import numpy as np

    from oracle_engine import OracleEngine
    from sentio_b200.retrievers import factory as factory_mod
    from sentio_b200.retrievers import sparse as sparse_mod

    monkeypatch.delenv("BM25_VARIANT", raising=False)
    monkeypatch.setattr(sparse_mod, "B200Engine", lambda device=0: OracleEngine())
    rng = np.random.default_rng(3)
    texts = [" ".join(f"w{rng.integers(0, 40)}" for _ in range(rng.integers(4, 30))) for _ in range(1500)]
    docs = [Document(id=f"doc-{i}", text=t, metadata={"source": f"s{i % 3}"}) for i, t in enumerate(texts)]
    a = sparse_mod.BM25Retriever(documents=docs, cache_dir=str(tmp_path))
    want = [(d.id, d.metadata["bm25_score"]) for d in a.retrieve("w1 w2 w2", top_k=20)]
    a.save()
    b = sparse_mod.BM25Retriever(cache_dir=str(tmp_path))
    assert b.load() is True
    assert [(d.id, d.metadata["bm25_score"]) for d in b.retrieve("w1 w2 w2", top_k=20)] == want
    foreign = str(tmp_path / "foreign.pkl")
    with open(foreign, "wb") as f:
        pickle.dump({"bm25": object(), "doc_ids": ["x"]}, f)
    assert b.load(foreign) is False and b.load(str(tmp_path / "none.pkl")) is False
    assert [(d.id, d.metadata["bm25_score"]) for d in b.retrieve("w1 w2 w2", top_k=20)] == want
    big = a.retrieve("w1 w2 w3 w4 w5 w6 w7 w8", top_k=1400)   # > 1024: device score dump + the reference's own cut
    assert 1024 < len(big) <= 1400 and [d.metadata["bm25_score"] for d in big] == sorted(
        (d.metadata["bm25_score"] for d in big), reverse=True)
    assert [d.id for d in big[:20]] == [d.id for d in a.retrieve("w1 w2 w3 w4 w5 w6 w7 w8", top_k=20)]
    assert a.retrieve("w1", top_k=0) == []

    # ---- _scroll_corpus: Qdrant payload schema {content, metadata} + string point ids, paged by 100
    class Point:
        def __init__(self, i, payload):
            self.id, self.payload = i, payload

    class Client:
        def __init__(self):
            self.calls = 0
            self.points = [Point(f"p{i}", {"content": f"text {i}", "metadata": {"page": i}}) for i in range(230)]
            self.points[7] = Point("p7", {"text": "from text key", "content": "ignored"})
            self.points[8] = Point("p8", None)                       # no payload: skipped (factory.py:110)
            self.points[9] = Point(9, {"page_content": "pc"})        # integer id -> str

        def scroll(self, collection_name, with_payload, with_vectors, limit, offset):
            self.calls += 1
            start = int(offset or 0)
            stop = min(len(self.points), start + limit)
            return self.points[start:stop], (stop if stop < len(self.points) else None)

    client = Client()
    got = factory_mod._scroll_corpus(client, "Sentio_docs")
    assert client.calls == 3 and len(got) == 229
    assert got[0].id == "p0" and got[0].text == "text 0" and got[0].metadata == {"page": 0}
    assert got[7].text == "from text key" and got[8].id == "9" and got[8].text == "pc" and got[8].metadata == {}


def test_global_bm25_stats_of_shards_equal_the_single_index(monkeypatch):
    """index.global_bm25_stats (the host half of HybridPipeline.build_bm25_sharded): per-shard (term, df) lists of 3
    contiguous shards -> the corpus-global idf / average idf / avgdl, bit-identical to the single-index build; and the
    chunk-seeded text generator returns the same docs whatever range is asked for."""
    import numpy as np

    from sentio_b200 import synth
    from sentio_b200.index import build_bm25_from_token_ids, global_bm25_stats

    flat, off = synth.text_corpus_tokens(5000, vocab=800)
    full = build_bm25_from_token_ids(flat, off)
    bounds = [(0, 1700), (1700, 3100), (3100, 5000)]
    parts = []
    for a, b in bounds:
        d = build_bm25_from_token_ids(flat[off[a]:off[b]], off[a:b + 1] - off[a])
        term_token = np.full(d.n_terms, -1, np.int64)
        known = np.nonzero(d.token_id_map >= 0)[0]
        term_token[d.token_id_map[known]] = known
        parts.append((term_token, np.diff(d.indptr), d.n_docs, int(d.doc_len.sum())))
    idf_of, avg_idf, n_docs, avgdl = global_bm25_stats([p[0] for p in parts], [p[1] for p in parts], [p[2] for p in parts],
                                                       [p[3] for p in parts], "okapi", 0.25)
    assert n_docs == 5000 and avgdl == full.avgdl and avg_idf == full.average_idf
    raw = np.nonzero(full.token_id_map >= 0)[0]
    assert [idf_of[int(t)] for t in raw] == [float(full.idf[full.token_id_map[t]]) for t in raw]
    a_flat, a_off = synth.text_corpus_tokens_range(0, 150_000)
    b_flat, b_off = synth.text_corpus_tokens_range(60_000, 140_000)
    assert np.array_equal(b_flat, a_flat[a_off[60_000]:a_off[140_000]])
    assert np.array_equal(b_off, a_off[60_000:140_001] - a_off[60_000])


def test_library_path_override(monkeypatch, tmp_path):
    """SENTIO_B200_LIB selects another build of the same sources (kernel A/B measurements); unset = the in-tree library."""
    import importlib

    import sentio_b200._lib as lib

    default = lib.LIB_PATH
    assert default.name == "libsentio_b200.so" and default.parent.name == "sentio_b200"
    # a reload rebinds the module's ctypes classes (SbCeConfig) and drops the loaded library, while engine.py keeps the
    # classes it imported: put the original namespace back so later engines in this process still match their prototypes
    saved = dict(vars(lib))
    monkeypatch.setenv("SENTIO_B200_LIB", str(tmp_path / "libsentio_b200_x.so"))
    try:
        assert importlib.reload(lib).LIB_PATH == tmp_path / "libsentio_b200_x.so"
    finally:
        monkeypatch.delenv("SENTIO_B200_LIB")
        try:
            assert importlib.reload(lib).LIB_PATH == default
        finally:
            vars(lib).clear()
            vars(lib).update(saved)
