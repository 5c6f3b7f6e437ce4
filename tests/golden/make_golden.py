"""Generate the committed golden fixtures by EXECUTING THE REFERENCE'S OWN MODULES (build container only).

    SENTIO_REFERENCE_ROOT=<checkout of chernistry/sentio> python tests/golden/make_golden.py [fixture ...]
                                              # writes tests/golden/<fixture>.json (default: all of them)

The reference's tests hold no numeric known answers for this path (SURVEY.md section 4), so the fixtures are outputs of
the unmodified reference code: HybridRetriever (src/core/retrievers/hybrid.py), BM25Retriever
(src/core/retrievers/sparse.py, on the rank_bm25 restatement), the scorer plugins (src/core/retrievers/scorers.py) and
JinaReranker's ordering / fallback logic (src/core/rerankers/jina_reranker.py).  Floats are stored with repr()
precision, i.e. bit-exact fp64.
"""
from __future__ import annotations

import json
import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import refload  # noqa: E402
from oracle import dense as dense_oracle  # noqa: E402


class HashEmbedder:
    """Deterministic embedder: unit-ish vector seeded by crc32(text) (stands in for the Jina embedder)."""

    def __init__(self, dim):
        self.dim = dim

    def embed_sync(self, text):
        rng = np.random.default_rng(zlib.crc32(text.strip().encode("utf-8")))
        v = rng.standard_normal(self.dim)
        return [float(x) for x in (v / np.linalg.norm(v)).astype(np.float32)]

    def embed_many_sync(self, texts):
        return [self.embed_sync(t) for t in texts]


class ListRetriever:
    def __init__(self, docs):
        self.docs = docs

    def retrieve(self, query, top_k=10):
        return self.docs[:top_k]


class ListPlugin:
    def __init__(self, hits):
        self.hits = hits

    def retrieve(self, query, top_k):
        return self.hits[:top_k]


class FixedScorer:
    def __init__(self, by_id):
        self.by_id = by_id

    def score(self, query, docs):
        return [self.by_id.get(d.id, 0.0) for d in docs]


def fusion_cases(ns):
    rng = np.random.default_rng(7)
    cases = []

    def run(name, method, rrf_k, dw, sw, dense, sparse, plugin, top_k, extras=None):
        # every sub-retriever is asked for top_k (hybrid.py:143,189,198): the fixture stores what they returned
        dense, sparse, plugin = dense[:top_k], sparse[:top_k], plugin[:top_k]
        D = ns.Document
        d_docs = [D(id=i, text=f"t{i}", metadata={"score": s}) for i, s in dense]
        s_docs = [D(id=i, text=f"t{i}", metadata={"bm25_score": s}) for i, s in sparse]
        scorers = [FixedScorer(e) for e in (extras or [])]
        hr = ns.HybridRetriever(dense_retriever=ListRetriever(d_docs), sparse_retriever=ListRetriever(s_docs),
                                rrf_k=rrf_k, scorer_plugins=scorers,
                                retriever_plugins=[ListPlugin(plugin)] if plugin else [], fusion_method=method,
                                dense_weight=dw, sparse_weight=sw)
        out = hr.retrieve("q", top_k=top_k)
        cases.append(dict(name=name, method=method, rrf_k=rrf_k, dense_weight=dw, sparse_weight=sw, dense=dense,
                          sparse=sparse, plugin=plugin, top_k=top_k, extras=extras or [],
                          expected=[[d.id, d.metadata["score"]] for d in out]))

    # the SURVEY section 8c known answers
    dense0 = [["A", 0.9], ["B", 0.8], ["C", 0.7]]
    sparse0 = [["D", 12.0], ["B", 7.0], ["E", 3.0]]
    run("survey_rrf", "rrf", 60, 0.5, 0.5, dense0, sparse0, [], 5)
    run("survey_wrrf", "weighted_rrf", 60, 0.7, 0.3, dense0, sparse0, [], 5)
    run("survey_comb", "comb_sum", 60, 0.7, 0.3, dense0, sparse0, [], 5)
    # randomised cases with overlaps, duplicates, plugin hits, scorer extras, truncation
    for c in range(24):
        n_d, n_s, n_p = int(rng.integers(0, 40)), int(rng.integers(0, 40)), int(rng.integers(0, 12))
        pool = [f"doc{j}" for j in range(60)]
        dense = [[str(rng.choice(pool)), float(rng.random())] for _ in range(n_d)]
        if c % 3 == 0:  # unique ids only (the normal case)
            seen = set()
            dense = [x for x in dense if not (x[0] in seen or seen.add(x[0]))]
        sparse_ids = list(rng.permutation(pool)[:n_s])
        sparse = [[str(i), float(rng.random() * 20)] for i in sparse_ids]
        if c % 5 == 0 and sparse:
            sparse = [[i, sparse[0][1]] for i, _ in sparse]  # all-equal -> normalises to 1.0
        plugin = [[str(rng.choice(pool + ["only_plugin_a", "only_plugin_b"])), float(rng.random())] for _ in range(n_p)]
        method = ["rrf", "weighted_rrf", "comb_sum"][c % 3]
        extras = []
        if c % 2 == 0:
            for _ in range(int(rng.integers(1, 4))):
                extras.append({i: float(rng.random()) for i in pool if rng.random() < 0.8})
        run(f"rand{c}", method, [60, 20, 1, 60.5][c % 4], float(rng.random()), float(rng.random()), dense, sparse,
            plugin, int(rng.integers(1, 50)), extras)
    return cases


def bm25_cases(ns):
    rng = np.random.default_rng(11)
    words = [f"w{j}" for j in range(40)] + ["The", "the", "Cat,", "cat", "dog.", "DOG"]
    cases = []
    for variant in ("okapi", "plus"):
        for c in range(4):
            n = [12, 60, 200, 35][c]
            p = np.arange(1, len(words) + 1) ** -1.1
            p /= p.sum()
            texts = [" ".join(rng.choice(words, size=int(rng.integers(3, 30)), p=p)) for _ in range(n)]
            if c == 3:  # pathological: a term in every doc (negative idf for okapi) + duplicate docs
                texts = ["common " + t for t in texts] + texts[:5]
                texts = [("common " + t) if not t.startswith("common") else t for t in texts]
            docs = [ns.Document(id=f"d{i}", text=t) for i, t in enumerate(texts)]
            os.environ["BM25_VARIANT"] = variant
            r = ns.BM25Retriever(documents=docs, variant=variant)
            queries = ["w0 w1 w2", "the cat", "w3 w3 w17 unknownword", "common w5", "zzz", "", "DOG dog. w0 w0 w0"]
            qcases = []
            for q in queries:
                scores = r.bm25.get_scores(q.lower().split())
                # stable tie order: the documented deviation from the reference's unstable np.argsort (sparse.py:180)
                order = np.argsort(-np.asarray(scores), kind="stable")[:10]
                exp = [[f"d{i}", float(scores[i])] for i in order if scores[i] > 0]
                res = r.retrieve(q, top_k=10)
                # the reference's own output must agree wherever it has no exact ties at the cut
                ref_pairs = [[d.id, d.metadata["bm25_score"]] for d in res]
                qcases.append(dict(query=q, scores=[float(s) for s in scores], top10=exp, reference_top10=ref_pairs))
            cases.append(dict(variant=variant, texts=texts, avgdl=r.bm25.avgdl,
                              idf={k: float(v) for k, v in r.bm25.idf.items()}, queries=qcases))
    os.environ.pop("BM25_VARIANT", None)
    return cases


def scorer_cases(ns):
    cases = []
    rng = np.random.default_rng(5)

    class Emb:
        def __init__(self, q, docs):
            self.q, self.docs = q, docs

        def embed_sync(self, text):
            return self.q

        def embed_many_sync(self, texts):
            return self.docs

    def run(name, q, docs, lam, w_mmr, w_sem):
        D = ns.Document
        dd = [D(id=str(i), text=f"t{i}") for i in range(len(docs))]
        emb = Emb(q, docs)
        mmr = ns.MMRScorer(emb, lambda_=lam, weight=w_mmr).score("q", dd)
        sem = ns.SemanticSimilarityScorer(emb, weight=w_sem).score("q", dd)
        cases.append(dict(name=name, q=q, docs=docs, lambda_=lam, w_mmr=w_mmr, w_sem=w_sem, mmr=mmr, sem=sem))

    q0 = [1.0, 0.0, 0.0]
    docs0 = [[0.9, 0.1, 0.0], [0.8, 0.2, 0.1], [0.0, 1.0, 0.0], [0.9, 0.1, 0.05]]
    run("survey_l05", q0, docs0, 0.5, 0.5, 0.8)
    run("survey_l07", q0, docs0, 0.7, 0.5, 0.8)
    for c in range(10):
        n, d = int(rng.integers(1, 40)), int(rng.choice([3, 16, 64, 200]))
        docs = rng.standard_normal((n, d)).astype(np.float32)
        if c % 3 == 0 and n > 2:
            docs[1] = docs[0]  # exact duplicate -> redundancy 1.0
        if c % 4 == 0 and n > 3:
            docs[2] = 0.0  # zero vector -> denom 0 branch
        q = rng.standard_normal(d).astype(np.float32)
        if c == 7:
            q = -docs[0]  # strongly negative relevances (break branch / clipping)
        run(f"rand{c}", [float(x) for x in q], [[float(x) for x in r] for r in docs],
            [0.0, 0.3, 0.5, 0.7, 1.0][c % 5], float(rng.random()), float(rng.random()))
    kw = ns.KeywordMatchScorer(weight=0.2).score(
        "What is machine learning?",
        [ns.Document(id="a", text="Machine learning is a subset of AI"),
         ns.Document(id="b", text="Deep learning uses neural networks")])
    return dict(semantic_mmr=cases, keyword=dict(query="What is machine learning?", weight=0.2,
                                                texts=["Machine learning is a subset of AI",
                                                       "Deep learning uses neural networks"], expected=kw))


class _StableArgsortNumpy:
    """numpy proxy whose argsort defaults to kind="stable".

    Documented deviation (DESIGN.md, SURVEY.md section 7 "tie semantics"): the reference's `np.argsort(-scores)`
    (sparse.py:180) is an unstable introsort, so its order among EXACT BM25 score ties is implementation defined; the
    fixtures (and the product) resolve such ties by ascending corpus position."""

    def __getattr__(self, name):
        return getattr(np, name)

    @staticmethod
    def argsort(a, *args, **kw):
        kw.setdefault("kind", "stable")
        return np.argsort(a, *args, **kw)


def hybrid_e2e_cases(ns):
    """Full reference stack: DenseRetriever over an exact-cosine Qdrant stand-in + BM25Retriever + HybridRetriever."""
    import src.core.retrievers.sparse as ref_sparse

    ref_sparse.np = _StableArgsortNumpy()
    rng = np.random.default_rng(21)
    dim = 64
    emb = HashEmbedder(dim)
    words = [f"w{j}" for j in range(300)]
    p = np.arange(1, 301) ** -1.07
    p /= p.sum()
    texts = [" ".join(rng.choice(words, size=int(rng.integers(8, 40)), p=p)) for _ in range(400)]
    vecs32 = np.asarray([emb.embed_sync(t) for t in texts], dtype=np.float32)
    rows16 = dense_oracle.stored_rows(vecs32)
    ids = [f"doc-{i}" for i in range(len(texts))]
    payloads = [{"content": t, "metadata": {"source": f"s{i % 7}"}} for i, t in enumerate(texts)]
    client = ns.NumpyQdrantClient()
    client.add_collection("Sentio_docs", rows16, ids, payloads)
    queries = [" ".join(rng.choice(words, size=6, p=p)) for _ in range(12)] + ["w0", "nothingmatches here"]
    out = dict(dim=dim, texts=texts, ids=ids, queries=queries, runs=[])
    for method in ("rrf", "weighted_rrf", "comb_sum"):
        for with_plugins in (False, True):
            corpus_docs = [ns.Document(id=i, text=t, metadata={"source": "corpus"}) for i, t in zip(ids, texts)]
            dense = ns.DenseRetriever(client=client, embedder=emb, collection_name="Sentio_docs")
            sparse = ns.BM25Retriever(documents=corpus_docs)
            plugins = None
            if with_plugins:
                plugins = [ns.SemanticSimilarityScorer(embedder=emb, weight=0.8), ns.KeywordMatchScorer(weight=0.2),
                           ns.MMRScorer(embedder=emb, lambda_=0.5, weight=0.5)]
            hr = ns.HybridRetriever(dense_retriever=dense, sparse_retriever=sparse, rrf_k=60, scorer_plugins=plugins,
                                    fusion_method=method, dense_weight=0.6, sparse_weight=0.4)
            res = []
            for q in queries:
                docs = hr.retrieve(q, top_k=15)
                res.append([[d.id, d.metadata["score"]] for d in docs])
            out["runs"].append(dict(method=method, plugins=with_plugins, results=res))
    return out


def hybrid_cache_cases(ns):
    """The reference stack with a POPULATED ``web_cache`` second collection (hybrid.py:146-182,208): cache hits are
    prepended to the dense hits, an id present in both lists accumulates twice (rrf) / keeps the last raw score
    (comb_sum dict semantics)."""
    import src.core.retrievers.sparse as ref_sparse

    ref_sparse.np = _StableArgsortNumpy()
    rng = np.random.default_rng(33)
    dim = 48
    emb = HashEmbedder(dim)
    words = [f"w{j}" for j in range(200)]
    p = np.arange(1, 201) ** -1.07
    p /= p.sum()
    texts = [" ".join(rng.choice(words, size=int(rng.integers(8, 30)), p=p)) for _ in range(300)]
    ids = [f"doc-{i}" for i in range(len(texts))]
    # the cache: 40 corpus documents under their corpus ids (duplicates across the two collections), 25 of them with an
    # edited text (different vector, same id), plus 30 web-only pages
    cache_texts, cache_ids = [], []
    for j, i in enumerate(rng.choice(len(texts), size=40, replace=False)):
        cache_ids.append(ids[int(i)])
        cache_texts.append(texts[int(i)] + (" cached copy" if j < 25 else ""))
    for j in range(30):
        cache_ids.append(f"web-{j}")
        cache_texts.append(" ".join(rng.choice(words, size=int(rng.integers(8, 30)), p=p)))
    client = ns.NumpyQdrantClient()
    client.add_collection("Sentio_docs", dense_oracle.stored_rows(np.asarray([emb.embed_sync(t) for t in texts], np.float32)),
                          ids, [{"content": t, "metadata": {"source": f"s{i % 5}"}} for i, t in enumerate(texts)])
    client.add_collection("web_cache", dense_oracle.stored_rows(np.asarray([emb.embed_sync(t) for t in cache_texts], np.float32)),
                          cache_ids, [{"content": t, "metadata": {"source": "web"}} for t in cache_texts])
    queries = [" ".join(rng.choice(words, size=5, p=p)) for _ in range(8)] + [cache_texts[3], texts[17], "w0"]
    out = dict(dim=dim, texts=texts, ids=ids, cache_texts=cache_texts, cache_ids=cache_ids, queries=queries, runs=[])
    os.environ["CACHE_COLLECTION_NAME"] = "web_cache"
    for method, with_plugins in (("rrf", False), ("weighted_rrf", False), ("comb_sum", False), ("rrf", True)):
        corpus_docs = [ns.Document(id=i, text=t, metadata={"source": "corpus"}) for i, t in zip(ids, texts)]
        dense = ns.DenseRetriever(client=client, embedder=emb, collection_name="Sentio_docs")
        sparse = ns.BM25Retriever(documents=corpus_docs)
        plugins = None
        if with_plugins:
            plugins = [ns.SemanticSimilarityScorer(embedder=emb, weight=0.8), ns.KeywordMatchScorer(weight=0.2),
                       ns.MMRScorer(embedder=emb, lambda_=0.5, weight=0.5)]
        hr = ns.HybridRetriever(dense_retriever=dense, sparse_retriever=sparse, rrf_k=60, scorer_plugins=plugins,
                                fusion_method=method, dense_weight=0.6, sparse_weight=0.4)
        assert hr._has_cache_collection
        res = []
        for q in queries:
            docs = hr.retrieve(q, top_k=12)
            res.append([[d.id, d.metadata["score"], d.text] for d in docs])
        out["runs"].append(dict(method=method, plugins=with_plugins, results=res))
    return out


def rerank_flow_cases(ns):
    """JinaReranker ordering / fallback behaviour with the HTTP call replaced by canned relevance scores."""
    from src.core.rerankers.jina_reranker import JinaReranker

    rr = JinaReranker(api_key="offline-key")
    cases = []
    rng = np.random.default_rng(3)
    for c in range(6):
        n = int(rng.integers(1, 12))
        rel = [float(x) for x in np.round(rng.random(n), 2)]  # rounding creates ties -> stable order matters
        docs = [ns.Document(id=f"r{i}", text=(f"text {i}" if i % 4 else ""), metadata={"content": f"fallback {i}"})
                for i in range(n)]
        top_k = int(rng.integers(1, 8))

        async def fake(query, doc_texts, tk, rel=rel):
            top_n = min(len(doc_texts), tk * 2)
            order = sorted(range(len(rel)), key=lambda i: rel[i], reverse=True)[:top_n]
            return {"results": [{"index": i, "relevance_score": rel[i]} for i in order]}

        rr._rerank_with_resilience = fake
        out = rr.rerank("some query", docs, top_k=top_k)
        cases.append(dict(kind="scores", rel=rel, top_k=top_k, n=n,
                          expected=[[d.id, d.metadata["rerank_score"], d.metadata["score"], d.text] for d in out]))
    docs = [ns.Document(id=f"r{i}", text=f"text {i}", metadata={"score": 0.5}) for i in range(4)]
    out = rr.rerank("   ", docs, top_k=3)
    cases.append(dict(kind="blank_query", n=4, top_k=3,
                      expected=[[d.id, d.metadata["rerank_score"], d.metadata["score"], d.text] for d in out]))
    return cases


def selector_cases(ns):
    """create_document_selector_node (nodes.py:231-372) on random candidate lists: score ties / missing / None scores,
    repeated ids, empty texts with and without the metadata["content"] fallback, blank texts, token budgets that cut the
    walk, the user_top_k override, reranked-vs-retrieved precedence."""
    from src.core.graph.nodes import create_document_selector_node
    from src.core.graph.state import create_initial_state

    rng = np.random.default_rng(11)
    cases = []
    for c in range(40):
        n = int(rng.integers(0, 14))
        docs = []
        for i in range(n):
            kind = int(rng.integers(0, 10))
            text = "x" * int(rng.integers(1, 400)) if kind < 8 else ("" if kind < 9 else "   ")
            meta = {}
            r = rng.random()
            if r < 0.7:
                meta["score"] = float(np.round(rng.random(), 1))  # rounding -> ties: the stable order matters
            elif r < 0.8:
                meta["score"] = None
            if rng.random() < 0.5:
                meta["content"] = "c" * int(rng.integers(0, 200))
            did = f"d{int(rng.integers(0, max(2, n - 2)))}" if rng.random() < 0.8 else ""
            docs.append(dict(id=did, text=text, metadata=meta))
        top_k = int(rng.integers(1, 8))
        max_tokens = int(rng.integers(20, 300))
        use_reranked = bool(rng.random() < 0.6)
        user_top_k = [None, 2, 5.0, "7"][int(rng.integers(0, 4))]
        state = create_initial_state("q")
        mk = lambda d: ns.Document(id=d["id"], text=d["text"], metadata=dict(d["metadata"]))
        state["retrieved_documents"] = [mk(d) for d in docs]
        if use_reranked:
            state["reranked_documents"] = [mk(d) for d in reversed(docs)]
        if user_top_k is not None:
            state["metadata"]["user_top_k"] = user_top_k
        out = create_document_selector_node(top_k=top_k, max_tokens=max_tokens)(state)
        cases.append(dict(docs=docs, top_k=top_k, max_tokens=max_tokens, use_reranked=use_reranked,
                          user_top_k=user_top_k,
                          selected=[[d.id, d.text, d.metadata] for d in out["selected_documents"]],
                          meta={k: v for k, v in out["metadata"].items() if k != "user_top_k"}))
    return cases


def reference_nodes_cases(ns):
    """The reference's retriever / reranker graph nodes (nodes.py:37-227), unmodified, driving THIS repository's
    HybridRetriever and B200Reranker on the oracle-backed engine double: the node outputs are what
    tests/test_reference_nodes.py holds the classes to."""
    sys.path.insert(0, os.path.dirname(HERE))
    from oracle_engine import OracleEngine
    from test_hybrid_e2e import _OracleStore

    import sentio_b200.retrievers.sparse as sparse_mod
    from sentio_b200.cross_encoder import CrossEncoderWeights
    from sentio_b200.document import Document
    from sentio_b200.rerankers.b200_reranker import B200Reranker
    from sentio_b200.retrievers.dense import DenseRetriever
    from sentio_b200.retrievers.hybrid import HybridRetriever
    from src.core.graph.nodes import create_reranker_node, create_retriever_node
    from src.core.graph.state import create_initial_state

    sparse_mod.B200Engine = lambda device=0: OracleEngine()
    os.environ.pop("BM25_VARIANT", None)
    dim, ce_seed, seq_len = 48, 3, 48
    texts = [f"topic{i % 9} w{i % 13} w{(i * 7) % 31} alpha{i % 5} chunk number {i}" for i in range(240)]
    ids = [f"doc-{i}" for i in range(len(texts))]
    queries = ["topic3 w4 alpha2", "w7 chunk", "nothing-in-the-vocabulary", "topic8 topic8 w30"]
    ce_cfg = dict(vocab_size=30522, hidden=128, layers=2, heads=4, intermediate=256, max_pos=64, type_vocab=2,
                  ln_eps=1e-12)
    emb = HashEmbedder(dim)
    payloads = [{"content": t, "metadata": {"source": f"s{i % 4}", "page": i}} for i, t in enumerate(texts)]
    store = _OracleStore(np.asarray(emb.embed_many_sync(texts), dtype=np.float32), ids, payloads)
    corpus = [Document(id=i, text=t, metadata={"source": "corpus"}) for i, t in zip(ids, texts)]
    eng = OracleEngine()
    hr = HybridRetriever(dense_retriever=DenseRetriever(client=store, embedder=emb, collection_name="Sentio_docs"),
                         sparse_retriever=sparse_mod.BM25Retriever(documents=corpus), rrf_k=60, scorer_plugins=[],
                         fusion_method="rrf", engine=eng)
    rr = B200Reranker(weights=CrossEncoderWeights.random(ce_cfg, seed=ce_seed), engine=eng, seq_len=seq_len)
    retrieve_node = create_retriever_node(hr, top_k=10)
    rerank_node = create_reranker_node(rr, top_k=4)

    def docs(lst):
        return [[d.id, d.text, dict(d.metadata)] for d in lst]

    cases = []
    for q in queries:
        state = retrieve_node(create_initial_state(q))
        case = dict(query=q, retrieved=docs(state["retrieved_documents"]), retrieve_metadata=dict(state["metadata"]))
        st5 = create_initial_state(q)
        st5["metadata"]["user_top_k"] = 5
        case["retrieved_user_top_k_5"] = [d.id for d in retrieve_node(st5)["retrieved_documents"]]
        state = rerank_node(state)
        case["reranked"] = docs(state["reranked_documents"])
        case["rerank_metadata"] = dict(state["metadata"])
        cases.append(case)

    class Boom:
        def retrieve(self, query, top_k=10):
            raise RuntimeError("index offline")

    raising = create_retriever_node(Boom(), top_k=3)(create_initial_state("q"))
    empty = rerank_node(create_initial_state("q"))
    return dict(dim=dim, texts=texts, ids=ids, payloads=payloads, ce_config=ce_cfg, ce_seed=ce_seed, seq_len=seq_len,
                retrieve_top_k=10, rerank_top_k=4, cases=cases,
                raising_retriever=dict(error="index offline", metadata=dict(raising["metadata"]),
                                       retrieved=docs(raising["retrieved_documents"])),
                no_documents=dict(metadata=dict(empty["metadata"]), reranked=docs(empty["reranked_documents"])))


FIXTURES = dict(fusion=fusion_cases, bm25=bm25_cases, scorers=scorer_cases, hybrid_e2e=hybrid_e2e_cases,
                hybrid_cache=hybrid_cache_cases, rerank_flow=rerank_flow_cases, selector=selector_cases,
                reference_nodes=reference_nodes_cases)


def main(names=None):
    ns = refload.load()
    fixtures = {name: FIXTURES[name](ns) for name in (names or FIXTURES)}
    for name, data in fixtures.items():
        path = os.path.join(HERE, f"{name}.json")
        with open(path, "w") as f:
            json.dump(data, f)
        print(name, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1:])
