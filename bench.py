#!/usr/bin/env python
"""bench.py -- retrieval queries/sec on BASELINE.json's configurations.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload dense|hybrid|rerank|bm25] [--batch B] [--inner R] [--n-docs N] [--dim D] [--top-k K]
                    [--rerank-k K2] [--shard auto|corpus|queries] [--no-extras] [--dump-outputs DIR]

Headline (`value`, `e2e`, `roofline`, `cpu_baseline`) = BASELINE.json configs[1]: 1 M docs x 1024-d, dense-only cosine
top_k=100 on 1 x B200.  A STEP = `--inner` R batches of `--batch` B queries per GPU through the hot path (defaults 64 x 256
dense, 32 x 128 hybrid, 2 x 64 rerank): R is chosen so that the K timed steps hold >= 1 s of device work, and is stated in
`config`.  The same JSON line carries, after the headline leg (unless --no-extras):

  workloads.hybrid      configs[2]  hybrid dense+BM25 rrf                       value / e2e / roofline.bm25 / cpu_baseline
  workloads.rerank      configs[3]  hybrid + cross-encoder rerank 100 -> 10     value / e2e / roofline.cross_encoder / cpu_baseline
  workloads.bm25_10k    configs[0]  10 k docs, BM25-only top_k=10: the reference CPU path (1024 queries) beside the GPU class
  latency_b1            HybridRetriever.retrieve(query, top_k=100) through the Document surface, one query at a time
  partitioned (N > 1)   the SAME 1 M corpus partitioned C = N ways (north_star's layout: corpus partition + ONE NCCL
                        all-gather of per-shard top-k): value, e2e and per-stage microseconds

Multi-GPU layout of the headline = C corpus shards x N/C query groups (--shard auto: the smallest C whose shard fits the
memory budget, 1 for the 2 GB corpus of the metric -> replicas, no collective).  Per-GPU work per step is constant in N
-> "scaling": "weak".

value   : whole-job queries/sec, inputs already resident in HBM (device entry points, CUDA-event timed, max over ranks)
e2e     : the same metric through the host-buffer C-ABI entry point (host queries -> H2D -> kernels -> D2H results)
roofline: dominant kernel (the dense scan) algorithmic bytes / CUDA-event duration vs MEASURED_PEAKS.json hbm_gbs
--dump-outputs DIR: after the timed steps, the headline leg's results of its LAST timed step (every batch of it, in order;
          rank 0) as DIR/<name>.npy, float64 (ids and counts are exact integers), at most 64 MB in all (larger outputs:
          a fixed, seeded sample of query rows, listed in DIR/query_rows.npy).  Inputs are seeded, so two builds run
          with the same arguments can be compared array for array.
cpu_baseline / --impl reference: the reference's CPU path (exact cosine in NumPy: fp32 `X @ q` with BLAS on a stated
          number of host threads + the best-first cut, both as the code base writes it -- full np.argsort,
          sparse.py:180 -- and with np.argpartition; BM25 via the rank_bm25 restatement) on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

_CORES = os.cpu_count() or 1
_BLAS_THREADS = min(_CORES, 64)
if "reference" in sys.argv or int(os.environ.get("WORLD_SIZE", "1")) == 1:
    # the CPU arms state their BLAS thread count instead of inheriting it (torchrun exports OMP_NUM_THREADS=1)
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(_BLAS_THREADS)

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "retrieval queries/sec @1M docs,1024-d,top_k=100"  # BASELINE.json metric (the workload actually run is in config)
UNIT = "queries/s"
DEFAULT_BATCH = {"dense": 256, "hybrid": 128, "rerank": 64, "bm25": 256}
DEFAULT_INNER = {"dense": 64, "hybrid": 32, "rerank": 2, "bm25": 64}
OUTPUT_NAMES = {"dense": ("ids", "scores", "counts"), "bm25": ("ids", "scores", "counts"),
                "hybrid": ("ids", "scores", "sources", "counts"), "rerank": ("ids", "scores", "counts")}
DUMP_LIMIT_BYTES = 64 << 20
NAMES = {"dense": "dense-only cosine", "hybrid": "hybrid dense+BM25 rrf", "bm25": "BM25-only",
         "rerank": "hybrid dense+BM25 rrf + cross-encoder rerank (MiniLM-L6 random-init)"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of every leg (the headline and each extra)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="dense", choices=["dense", "hybrid", "rerank", "bm25"])
    ap.add_argument("--rerank-k", type=int, default=10, help="documents kept after the cross-encoder (config 4: 100 -> 10)")
    ap.add_argument("--batch", type=int, default=None, help="queries per batch PER GPU (256 dense, 128 hybrid, 64 rerank)")
    ap.add_argument("--inner", type=int, default=None,
                    help="batches per step (64 dense, 32 hybrid, 2 rerank): sized for >= 1 s of timed device work")
    ap.add_argument("--n-docs", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--top-k", type=int, default=100)
    ap.add_argument("--cpu-sample", type=int, default=24, help="queries in the bounded CPU-baseline sample (0 = skip)")
    ap.add_argument("--no-extras", action="store_true",
                    help="headline leg only (skip workloads.* / latency_b1 / partitioned)")
    ap.add_argument("--extras", default="hybrid,rerank,bm25_10k,latency_b1,partitioned",
                    help="comma list of the extra legs run after a default dense headline")
    ap.add_argument("--shard", default="auto", choices=["auto", "corpus", "queries"],
                    help="--gpus N > 1 layout = C corpus shards x N/C query groups.  'corpus': C = N (contiguous doc ranges "
                         "+ ONE NCCL all-gather of per-shard top-k, north_star's layout for corpora that must be "
                         "partitioned); 'queries': C = 1 (corpus replicated, queries split, no collective); 'auto' "
                         "(default): the smallest C whose shard fits --gpu-mem-budget-gb")
    ap.add_argument("--corpus-shards", type=int, default=0, help="explicit C (must divide N); overrides --shard")
    ap.add_argument("--gpu-mem-budget-gb", type=float, default=64.0,
                    help="HBM one GPU may spend on index data under --shard auto (B200: 180 GB)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the headline leg's results of its last timed step to DIR/<name>.npy (<= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p.get("bf16_tflops_sustained", 1429.5)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md: 6.65 TB/s, 1.4 PF sustained bf16)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.device), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


def workload_name(n_docs, dim, kind, top_k, rerank_k):
    return (f"{n_docs}-doc synthetic, {dim}-d, {NAMES[kind]} top_k={top_k}" + (f"->{rerank_k}" if kind == "rerank" else ""))


# --------------------------------------------------------------------------------------------- synthetic workload
class Workload:
    """Synthetic corpus / queries (SURVEY Appendix C), generated lazily: the text side only when a leg needs it.
    Corpora above 2 M docs are generated shard-locally from independently seeded chunks (synth.dense_corpus_range), so
    a rank only ever materialises its own rows."""

    def __init__(self, n_docs, dim):
        self.n_docs, self.dim = n_docs, dim
        self.gen_s = 0.0
        self._x16 = {}
        self._text = None
        from sentio_b200 import synth

        self.synth = synth
        self.q = synth.query_vectors(1024, dim)
        self.q_tokens = synth.query_tokens(1024)

    def rows(self, lo, hi):
        key = (lo, hi)
        if key not in self._x16:
            t0 = time.time()
            if self.n_docs > 2_000_000:
                x = self.synth.dense_corpus_range(lo, hi, self.dim)
            else:
                full = self._x16.get((0, self.n_docs))
                if full is None:
                    full = self.synth.dense_corpus(self.n_docs, self.dim)
                    self._x16[(0, self.n_docs)] = full
                x = full[lo:hi]
            self._x16[key] = x
            self.gen_s += time.time() - t0
        return self._x16[key]

    def text(self):
        if self._text is None:
            t0 = time.time()
            self._text = (self.synth.text_corpus_tokens_range(0, self.n_docs) if self.n_docs > 2_000_000 else
                          self.synth.text_corpus_tokens(self.n_docs))   # > 2 M docs: the chunk-seeded corpus of the shards
            self.gen_s += time.time() - t0
        return self._text

    def text_range(self, lo, hi):
        """(flat, off) of docs [lo, hi), shard-local offsets: a slice of the corpus up to 2 M docs, generated shard-locally
        (independently seeded chunks) above."""
        t0 = time.time()
        if self.n_docs > 2_000_000:
            out = self.synth.text_corpus_tokens_range(lo, hi)
        else:
            flat, off = self.text()
            out = (flat[off[lo]:off[hi]], off[lo:hi + 1] - off[lo])
        self.gen_s += time.time() - t0
        return out


# --------------------------------------------------------------------------------------------- CPU reference arm
def cpu_reference(kind, wl: Workload, n_queries, top_k, rerank_k):
    """Times the reference's CPU path on this box's host cores on a bounded sample of the same workload."""
    from oracle import dense as dense_oracle

    x16 = wl.rows(0, wl.n_docs)
    x32 = x16.astype(np.float32)
    x32 /= np.linalg.norm(x32, axis=1, keepdims=True)  # Qdrant normalises at upsert; the scan is then a plain dot
    q = wl.q
    fast = ce_model = None
    if kind in ("hybrid", "rerank"):
        from oracle import fusion as fusion_oracle
        from oracle.rank_bm25_port import FastBM25
        from sentio_b200.index import build_bm25_from_token_ids

        flat, off = wl.text()
        if getattr(wl, "_host_idx", None) is None:   # the reference-side index build is not part of the timed queries
            wl._host_idx = build_bm25_from_token_ids(flat, off)
        idx = wl._host_idx
        fast = FastBM25(idx.indptr, idx.post_doc, idx.post_tf, idx.doc_len, idx.idf, idx.avgdl)
        terms = [idx.term_ids(t) for t in wl.q_tokens]
    if kind == "rerank":
        from oracle import cross_encoder as ce_oracle
        from sentio_b200.cross_encoder import MINILM_L6
        from sentio_b200.index import hash_tokenize_pairs

        ce_model = ce_oracle.hf_model(MINILM_L6, seed=0)
    for i in range(2):  # warm-up
        dense_oracle.fast_topk_f32(x32, q[i], top_k)
    t0 = time.perf_counter()
    for i in range(n_queries):
        di, ds = dense_oracle.fast_topk_f32(x32, q[i % len(q)], top_k)
        if fast is not None:
            s = fast.get_scores(list(terms[i % len(terms)]))
            order = np.argsort(-s)[:top_k]
            sp = [(int(j), float(s[j])) for j in order if s[j] > 0]
            fused = fusion_oracle.fuse("rrf", 60, 0.5, 0.5, [(int(a), float(b)) for a, b in zip(di, ds)], sp, [], top_k)
            if ce_model is not None:
                flat, off = wl.text()
                qtext = wl.synth.token_text(wl.q_tokens[i % len(terms)])
                texts = [wl.synth.token_text(flat[off[d]:off[d + 1]]) for d, _, _ in fused]
                ids, tt, lens = hash_tokenize_pairs(qtext, texts, 128)
                _, sig = ce_oracle.hf_scores(ce_model, ids, tt, lens, batch=len(texts))
                sorted(range(len(sig)), key=lambda j: -sig[j])[:rerank_k]
    dt = time.perf_counter() - t0
    out = {"value": n_queries / dt, "unit": UNIT, "cores": _BLAS_THREADS, "host_cpus": _CORES, "kind": "port",
           "sample": (f"{n_queries} queries of the same workload; dense = fp32 X@q (NumPy/BLAS, {_BLAS_THREADS} threads "
                      f"set explicitly) + np.argsort[:k] (the cut as the reference writes it, sparse.py:180)"
                      + ("; BM25 = CSR restatement of rank_bm25 get_scores + np.argsort; rrf fusion in Python" if fast else "")
                      + ("; rerank = HuggingFace BertForSequenceClassification (MiniLM-L6 shape) fp32 on CPU, 100 pairs/query"
                         if ce_model is not None else ""))}
    if kind == "dense":   # the same scan with a partial sort: what a tuned NumPy implementation would do
        t0 = time.perf_counter()
        for i in range(n_queries):
            s = x32 @ q[i % len(q)]
            part = np.argpartition(-s, top_k)[:top_k]
            part[np.argsort(-s[part])]
        out["value_argpartition"] = n_queries / (time.perf_counter() - t0)
    return out, dt / n_queries


def bm25_10k_leg(device, top_k=10, n_queries=1024):
    """BASELINE configs[0]: 10 k docs, BM25-only top_k = 10.  The reference CPU path (rank_bm25's dict-based get_scores
    as restated in oracle/, np.argsort, score > 0 filter -- sparse.py:159-203) over all 1024 queries, beside the GPU
    BM25Retriever arrays path on the same corpus and queries, ids compared."""
    from oracle.rank_bm25_port import BM25Okapi
    from sentio_b200 import synth
    from sentio_b200.document import Document
    from sentio_b200.retrievers.sparse import BM25Retriever

    n = 10_000
    flat, off = synth.text_corpus_tokens(n)
    texts = [synth.token_text(flat[off[i]:off[i + 1]]) for i in range(n)]
    queries = [synth.token_text(t) for t in synth.query_tokens(n_queries)]
    ref = BM25Okapi([t.lower().split() for t in texts])
    t0 = time.perf_counter()
    want = []
    for qtext in queries:
        s = ref.get_scores(qtext.lower().split())
        order = np.argsort(-s, kind="stable")[:top_k]
        want.append([int(i) for i in order if s[i] > 0])
    cpu_s = time.perf_counter() - t0
    os.environ.pop("BM25_VARIANT", None)
    r = BM25Retriever(documents=[Document(id=str(i), text=t) for i, t in enumerate(texts)], device=device)
    r.retrieve_batch_arrays(queries[:64], top_k)
    t0 = time.perf_counter()
    ids, sc, cnt = r.retrieve_batch_arrays(queries, top_k)
    gpu_s = time.perf_counter() - t0
    same = all([int(x) for x in ids[b, :cnt[b]]] == want[b] for b in range(n_queries))
    t0 = time.perf_counter()
    for qtext in queries[:128]:
        r.retrieve(qtext, top_k=top_k)
    one_s = (time.perf_counter() - t0) / 128
    return {"workload": f"{n}-doc synthetic, 768-d (unused: BM25-only), top_k={top_k}, {n_queries} queries",
            "cpu_reference_qps": n_queries / cpu_s, "cpu_kind": "port (rank_bm25 0.2.2 restatement, 1 thread: pure Python)",
            "gpu_batch_qps": n_queries / gpu_s, "gpu_retrieve_one_by_one_qps": 1.0 / one_s,
            "ids_identical_to_reference_path": bool(same), "unit": UNIT}


# --------------------------------------------------------------------------------------------- one timed leg
class Leg:
    """One workload on one pipeline: the device-resident timed region and the host-buffer (e2e) timed region."""

    def __init__(self, kind, pipe, wl: Workload, args, world, rank, local_rank, C, my_group, lo, hi, idx, rerank_state):
        import torch

        self.torch = torch
        self.kind, self.pipe, self.wl, self.args = kind, pipe, wl, args
        self.world, self.rank, self.local_rank, self.C, self.my_group = world, rank, local_rank, C, my_group
        self.lo, self.hi, self.idx = lo, hi, idx
        self.eng = pipe.engine
        self.dev = f"cuda:{local_rank}"
        self.k = args.top_k
        self.B_gpu = args.batch if kind == args.workload and args.batch else DEFAULT_BATCH[kind]
        self.inner = args.inner if kind == args.workload and args.inner else DEFAULT_INNER[kind]
        self.B = self.B_gpu * C                     # queries this rank scores per batch (all C ranks of a group: the same)
        self.B_total = self.B_gpu * world           # queries per batch over the whole job
        self.q_shift = my_group * self.B
        self.q_all = torch.from_numpy(wl.q).to(self.dev)
        self.n_q = self.q_all.shape[0]
        self.term_lists = [idx.term_ids(t) for t in wl.q_tokens] if idx is not None else None
        self.q_tok_all = rerank_state["q_tok_all"] if rerank_state else None
        self.ring = max(1, min(8, self.n_q // max(1, self.B_total)))   # distinct batches (1024 seeded queries, cycled)

    # ---- inputs
    def batch_ids(self, j):
        s = (j * self.B_total + self.q_shift) % self.n_q
        return [(s + i) % self.n_q for i in range(self.B)]

    def dev_inputs(self, j):
        torch, ids = self.torch, self.batch_ids(j)
        qt = self.q_all[ids].contiguous()
        if self.kind == "dense":
            return (qt,)
        flat, off = self.eng.pack_queries([self.term_lists[i] for i in ids])
        base = (qt, torch.from_numpy(flat).to(self.dev), torch.from_numpy(off).to(self.dev), int(off[-1]),
                int(np.diff(off).max()))
        if self.kind != "rerank":
            return base
        qtok = torch.from_numpy(self.q_tok_all[ids]).to(self.dev)
        qlen = torch.full((self.B,), self.q_tok_all.shape[1], dtype=torch.int32, device=self.dev)
        return base + (qtok, qlen)

    def run_dev(self, inp):
        p, k, a = self.pipe, self.k, self.args
        if self.kind == "dense":
            return p.dense_dev(inp[0], k)
        if self.kind == "bm25":
            return p.engine.bm25_topk_dev(inp[1], inp[2], self.B, inp[3], inp[4], k)
        if self.kind == "rerank":
            return p.hybrid_rerank_dev(inp[0], inp[1], inp[2], inp[3], inp[4], inp[5], inp[6], k, a.rerank_k, 128, "rrf",
                                       60, 0.5, 0.5)
        return p.hybrid_dev(inp[0], inp[1], inp[2], inp[3], inp[4], k, "rrf", 60, 0.5, 0.5)

    def run_host(self, j):
        p, k, a = self.pipe, self.k, self.args
        ids = self.batch_ids(j)
        q = self.host_q[j % self.ring]
        if self.kind == "dense":
            return p.search_dense(q, k, out=self.host_out[j % len(self.host_out)] if self.host_out else None)
        terms = self.host_terms[j % self.ring]
        if self.kind == "bm25":
            return p.engine.bm25_topk(terms, k)
        if self.kind == "rerank":
            return p.search_hybrid_rerank(q, terms, self.q_tok_all[ids], np.full(self.B, self.q_tok_all.shape[1], np.int32),
                                          k, a.rerank_k, 128, "rrf", 60, 0.5, 0.5)
        return p.search_hybrid(q, terms, k, "rrf", 60, 0.5, 0.5)

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist

            dist.barrier()
        self.torch.cuda.synchronize()

    def _max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            import torch.distributed as dist

            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- the two timed regions
    def run(self, steps, warmup, sample_clocks=True, capture=False):
        """``capture``: also keep every batch result of the last timed step (device copies, ``outputs``)."""
        torch, eng = self.torch, self.eng
        inputs = [self.dev_inputs(j) for j in range(self.ring)]
        for s in range(warmup):
            for r in range(self.inner):
                self.run_dev(inputs[(s * self.inner + r) % self.ring])
        self.barrier()
        eng.profile(True)
        if self.kind == "rerank":
            eng.ce_stats(reset=True)
        launches0 = eng.launch_count()
        sampler = ClockSampler(self.local_rank)
        if self.rank == 0 and sample_clocks:
            sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        outputs = None
        try:
            self.barrier()
            ev0.record()
            for s in range(steps):
                for r in range(self.inner):
                    out = self.run_dev(inputs[(s * self.inner + r) % self.ring])
                    if capture and s == steps - 1:   # the path reuses its output buffers: copy each batch aside
                        if outputs is None:
                            outputs = [torch.empty((self.inner, *t.shape), dtype=t.dtype, device=t.device) for t in out]
                        for o, t in zip(outputs, out):
                            o[r].copy_(t)
            ev1.record()
            self.barrier()
        finally:
            clocks = sampler.stop() if (self.rank == 0 and sample_clocks) else None
        ms_total = ev0.elapsed_time(ev1)
        launches = eng.launch_count() - launches0
        prof = {name: eng.profile_read(name) for name in ("dense_scan", "dense_merge", "dense_sample", "bm25_score",
                                                          "bm25_select", "fuse", "ce")}
        ce_stats = eng.ce_stats() if self.kind == "rerank" else (0, 0, 0)
        eng.profile(False)
        ms_total = self._max_over_ranks(ms_total)
        n_batches = steps * self.inner
        value = self.B_total * n_batches / (ms_total / 1e3)

        # e2e: host buffers in, host results out, every batch
        # the caller's request / response buffers: page-locked and reused (a serving loop's I/O rings), so the library
        # copies straight between them and the device
        self.host_q, self.host_out = [], []
        for j in range(self.ring):
            src = self.wl.q[self.batch_ids(j)]
            if self.world == 1 and self.kind == "dense" and hasattr(eng, "pinned_empty"):
                buf = eng.pinned_empty(src.shape, np.float32)
                buf[...] = src
                self.host_q.append(buf)
                self.host_out.append((eng.pinned_empty((self.B, self.k), np.int64),
                                      eng.pinned_empty((self.B, self.k), np.float64), eng.pinned_empty((self.B,), np.int32)))
            else:
                self.host_q.append(src)
        self.host_terms = None
        if self.term_lists is not None:
            self.host_terms = [[self.term_lists[i] for i in self.batch_ids(j)] for j in range(self.ring)]
        for s in range(min(warmup, 2) * self.inner):
            self.run_host(s)
        self.barrier()
        t0 = time.perf_counter()
        for s in range(n_batches):
            self.run_host(s)
        self.barrier()
        e2e_s = self._max_over_ranks(time.perf_counter() - t0)
        B, k, a = self.B, self.k, self.args
        h2d = B * a.dim * 4 if self.kind != "bm25" else 0
        d2h = B * k * 16 + B * 4
        if self.term_lists is not None:
            h2d += sum(len(x) for x in self.host_terms[0]) * 4 + (B + 1) * 4
            d2h += B * k * 4 if self.kind != "bm25" else 0
        if self.kind == "rerank":
            h2d += B * self.q_tok_all.shape[1] * 4 + B * 4
            d2h = self.B_gpu * a.rerank_k * 12 + self.B_gpu * 4  # every rank returns the rows of the queries it reranked
        e2e = {"value": self.B_total * n_batches / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d * self.world * self.inner,
               "d2h_bytes_per_step": d2h * self.world * self.inner,
               "timer": "host wall clock around the public host-buffer calls of the step (H2D, kernels, D2H, one sync "
                        "per call); bytes are summed over ranks and over the step's batches",
               "host_buffers": "page-locked request / response arrays reused across calls (engine.pinned_empty)"
                               if self.host_out else "pageable NumPy arrays (staged through the library's pinned buffers)"}
        return {"value": value, "ms_total": ms_total, "ms_per_step": ms_total / steps, "steps": steps, "n_batches": n_batches,
                "clocks": clocks, "launches": int(launches), "prof": prof, "ce_stats": ce_stats, "e2e": e2e,
                "timed_region_s": ms_total / 1e3, "outputs": outputs}

    # ---- rooflines
    def roofline_dense(self, res):
        hbm, _, src = peaks()
        rows = self.hi - self.lo
        n_pad = (rows + 127) // 128 * 128
        d_pad = (self.args.dim + 7) // 8 * 8
        alg = n_pad * d_pad * 2 + n_pad * 4
        n_scan, scan_ms = res["prof"]["dense_scan"]
        avg = scan_ms / max(n_scan, 1)
        ach = alg / (avg * 1e-3) / 1e9 if n_scan else 0.0
        qpl = (self.B * res["n_batches"]) / max(n_scan, 1)
        kern = ("dense_scan_mma2_kernel (tcgen05 cta_group::2 pair, 128 queries per pass)" if qpl > 64 else
                "dense_scan_mma_kernel (tcgen05, <= 64 queries per pass)" if self.B >= 16 else "dense_scan_kernel (FFMA2)")
        out = {"bound": "hbm", "kernel": kern, "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
               "traffic": None, "traffic_source": None, "peak_source": src, "algorithmic_bytes_per_launch": alg,
               "avg_launch_ms": avg, "launches_timed": n_scan, "queries_per_launch": qpl,
               "share_of_step": scan_ms / res["ms_total"],
               "other_dense_stages_ms_per_batch": {
                   "sampling_passes+threshold_select": res["prof"]["dense_sample"][1] / max(res["n_batches"], 1),
                   "window_select+fp64_rescore": res["prof"]["dense_merge"][1] / max(res["n_batches"], 1)}}
        prof = os.path.join(ROOT, "profiles", "r02_dense_scan_ncu.json")
        if os.path.exists(prof) and self.C == 1:
            try:
                out["traffic"] = json.load(open(prof)).get("dram_bytes_per_launch")
                out["traffic_source"] = "profiles/r02_dense_scan_ncu.json (ncu --set full of the same kernel, static)"
            except Exception:
                pass
        return out

    def roofline_bm25(self, res):
        hbm, _, _ = peaks()
        n_bm, bm_ms = res["prof"]["bm25_score"]
        if not n_bm or self.idx is None:
            return None
        sidx = self.idx   # C > 1: a shard-local index (pipeline.build_bm25_sharded), its df are the shard's
        df = np.diff(sidx.indptr)
        postings = 0
        for j in range(self.ring):
            for i in self.batch_ids(j):
                t = self.term_lists[i]
                postings += int(df[t[t >= 0]].sum())
        postings = postings * res["n_batches"] / self.ring
        return {"bound": "latency + l1tex", "kernel": "bm25_range_kernel (sample + collect)",
                "postings_per_s": postings / (bm_ms * 1e-3), "postings_per_query": postings / (self.B * res["n_batches"]),
                "algorithmic_bytes": postings * 12, "posting_GBps": postings * 12 / (bm_ms * 1e-3) / 1e9,
                "frac_of_hbm_peak_if_every_posting_came_from_dram": postings * 12 / (bm_ms * 1e-3) / 1e9 / hbm,
                "ms_total": bm_ms, "share_of_step": bm_ms / res["ms_total"],
                "note": "the posting lists shared by a batch are served by L2 (ncu: DRAM traffic << posting bytes); ncu of the "
                        "collect pass (profiles/r02_run13_bm25_range_ncu.md): issue slots 55 % busy, L1TEX 69 %, a third of "
                        "the stalls on load latency -- no single limiter, so postings/s is the figure of merit, not GB/s"}

    def roofline_ce(self, res):
        _, tpeak, _ = peaks()
        n_ce, ce_ms = res["prof"]["ce"]
        if not n_ce:
            return None
        ce_pairs, ce_rows, ce_sq = res["ce_stats"]
        flops = 6 * (24 * 384 * 384 * ce_rows + 4 * 384 * ce_sq)
        tf = flops / (ce_ms * 1e-3) / 1e12
        return {"bound": "tensor", "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": tf / tpeak, "ms_total": ce_ms,
                "forward_calls": n_ce, "pairs": ce_pairs, "mean_pair_len": ce_rows / max(ce_pairs, 1),
                "flops_counted": "L*(24*H^2*sum(len) + 4*H*sum(len^2)), padding excluded",
                "share_of_step": ce_ms / res["ms_total"]}


def latency_b1(pipe, wl: Workload, idx, n_queries=200, top_k=100):
    """The call the graph makes: HybridRetriever.retrieve(query, top_k=100), one query at a time, through the Document
    surface (DenseRetriever over a vector-store facade on the loaded index + BM25Retriever on the loaded postings)."""
    from sentio_b200.document import Document
    from sentio_b200.retrievers.dense import DenseRetriever
    from sentio_b200.retrievers.hybrid import HybridRetriever
    from sentio_b200.retrievers.sparse import BM25Retriever
    from sentio_b200.vector_store import ScoredPoint

    import dataclasses

    synth, eng = wl.synth, pipe.engine
    # text queries need a token-string vocabulary (the device-built index of the integer corpus only maps raw token ids)
    idx = dataclasses.replace(idx, vocab={f"w{raw}": int(t) for raw, t in enumerate(idx.token_id_map) if t >= 0})

    def text_of(i):   # placeholder document text: the synthetic corpus has token ids, not strings, and rendering 80 tokens
        return f"synthetic document {i}"   # per hit would time str.join, not the retrieval surface

    class Store:   # QdrantClient-shaped facade over the ALREADY loaded dense index (no second 2 GB copy)
        def collection_exists(self, collection_name):
            return collection_name == "Sentio_docs"

        def search(self, collection_name, query_vector, limit=10, with_payload=True, with_vectors=False, **kw):
            ids, sc, cnt = eng.dense_topk(np.asarray(query_vector, np.float32).reshape(1, -1), int(limit))
            return [ScoredPoint(id=str(int(ids[0, j])), score=float(sc[0, j]),
                                payload={"content": text_of(int(ids[0, j])), "metadata": {"source": "synthetic"}})
                    for j in range(int(cnt[0]))]

    class Embedder:  # the query embedding forward is a separate row (SURVEY 8f-1); here a table of seeded unit vectors
        def __init__(self):
            self.at = {}

        def embed_sync(self, text):
            return self.at[text]

    class DocMap:    # materialises a corpus Document on demand (1 M Python objects up front would measure the allocator)
        def get(self, doc_id, default=None):
            return Document(id=doc_id, text=text_of(int(doc_id)), metadata={"source": "synthetic"})

    class DocIds:
        def __getitem__(self, row):
            return str(row)

    emb = Embedder()
    sparse = BM25Retriever(device=pipe.device)
    sparse.bm25, sparse.doc_ids, sparse.doc_map, sparse._engine = idx, DocIds(), DocMap(), eng
    dense = DenseRetriever(client=Store(), embedder=emb, collection_name="Sentio_docs")
    hr = HybridRetriever(dense_retriever=dense, sparse_retriever=sparse, rrf_k=60, scorer_plugins=[], fusion_method="rrf",
                         engine=eng)
    texts = [synth.token_text(t) for t in wl.q_tokens[:n_queries + 8]]
    for i, t in enumerate(texts):
        emb.at[t] = wl.q[i]
    out = {}
    for name, fn in (("hybrid", lambda t: hr.retrieve(t, top_k=top_k)), ("dense", lambda t: dense.retrieve(t, top_k=top_k))):
        for t in texts[:8]:
            fn(t)
        lat = []
        for t in texts[8:]:
            t0 = time.perf_counter()
            docs = fn(t)
            lat.append(time.perf_counter() - t0)
        lat = np.asarray(lat) * 1e3
        out[name] = {"p50_ms": float(np.percentile(lat, 50)), "p99_ms": float(np.percentile(lat, 99)),
                     "mean_ms": float(lat.mean()), "queries": len(lat), "docs_returned": len(docs)}
    out["call"] = (f"HybridRetriever.retrieve(query, top_k={top_k}) / DenseRetriever.retrieve, B = 1, Document objects out "
                   "(placeholder document texts; query embedding = table lookup)")
    return out


def dump_outputs(path, kind, outputs):
    """The last timed step's results as <path>/<name>.npy: [batches_per_step * queries_per_batch, ...] rows in the order
    the step ran them, float64 (float32 arrays stay float32).  Above DUMP_LIMIT_BYTES a fixed, seeded sample of rows is
    kept and its row numbers go to query_rows.npy."""
    arrays = []
    for name, t in zip(OUTPUT_NAMES[kind], outputs):
        a = t.cpu().numpy()
        a = a.reshape(-1, *a.shape[2:])
        arrays.append((name, a if a.dtype == np.float32 else a.astype(np.float64)))
    rows = arrays[0][1].shape[0]
    row_bytes = sum(a.nbytes for _, a in arrays) // max(rows, 1)
    if rows * row_bytes > DUMP_LIMIT_BYTES - (1 << 20):
        keep = (DUMP_LIMIT_BYTES - (1 << 20)) // (row_bytes + 8)
        sel = np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
        arrays = [(name, a[sel]) for name, a in arrays] + [("query_rows", sel.astype(np.float64))]
    os.makedirs(path, exist_ok=True)
    for name, a in arrays:
        np.save(os.path.join(path, f"{name}.npy"), a)


# --------------------------------------------------------------------------------------------- main
_RESULT_OUT = sys.stdout


def _emit(line):
    """The ONE JSON line of the contract, on the process's original stdout."""
    _RESULT_OUT.write(json.dumps(line) + "\n")
    _RESULT_OUT.flush()


def main():
    args = parse_args()
    # Libraries print to stdout behind our back (NCCL's "NCCL version ..." banner at communicator creation): keep a private
    # handle on the real stdout for the result line and point fd 1 at stderr for everything else.
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    kind = args.workload
    B_gpu = args.batch or DEFAULT_BATCH[kind]
    inner = args.inner or DEFAULT_INNER[kind]
    name = workload_name(args.n_docs, args.dim, kind, args.top_k, args.rerank_k)
    est_gb = args.n_docs * args.dim * 2 / 1e9 + (args.n_docs * 60 * 12 / 1e9 if kind != "dense" else 0.0)
    from sentio_b200.pipeline import plan_layout

    try:
        C, _ = plan_layout(world, est_gb, args.shard, args.corpus_shards, args.gpu_mem_budget_gb)
    except ValueError as exc:
        raise SystemExit(str(exc))
    n_groups, my_group, r_in = world // C, rank // C, rank % C
    config = {"workload": name, "queries_per_batch_per_gpu": B_gpu, "batches_per_step": inner,
              "batch_queries_per_step": B_gpu * world * inner, "store_dtype": "fp16", "shards": C, "query_groups": n_groups,
              "index_gb_estimate": round(est_gb, 2),
              "multi_gpu": ("single GPU" if world == 1 else
                            f"{C} corpus shard(s) x {n_groups} query group(s): "
                            + ("corpus partition + one NCCL all-gather of per-shard top-k" if C > 1 else
                               "corpus replicated, no collective")
                            + ("; queries split across groups" if n_groups > 1 else "")
                            + (f" [--corpus-shards {C}]" if args.corpus_shards else f" [--shard {args.shard}]")),
              "l2_policy": "corpus (2.05 GB) is larger than L2 (126 MB); no flush needed",
              "query_set": "1024 seeded unit vectors, cycled"}

    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the results of the GPU path: use it with --impl b200")
        if rank != 0:
            return 0
        wl = Workload(args.n_docs, args.dim)
        per_step = max(1, min(B_gpu, 4))
        total = per_step * (args.steps + args.warmup)
        base, per_q = cpu_reference(kind if kind != "bm25" else "dense", wl, total, args.top_k, args.rerank_k)
        line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_q * per_step * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": {**config, "batch_queries_per_step": per_step, "batches_per_step": 1,
                                                "queries_per_batch_per_gpu": per_step},
                "cpu_baseline": {**base, "sample": f"{per_step} queries per step; " + base["sample"]},
                "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        _emit(line)
        return 0

    import torch
    import torch.distributed as dist

    from sentio_b200.pipeline import HybridPipeline

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    n = args.n_docs
    lo, hi = ((n * r_in) // C, (n * (r_in + 1)) // C) if C > 1 else (0, n)
    wl = Workload(n, args.dim)
    groups = {}

    def group_for(c):   # one NCCL communicator per corpus group (every rank creates all of them, in order)
        if c == 1 or c in groups:
            return groups.get(c)
        mine = None
        if c == world:
            mine = dist.group.WORLD
        else:
            for g in range(world // c):
                pg = dist.new_group(list(range(g * c, (g + 1) * c)))
                if g == rank // c:
                    mine = pg
        groups[c] = mine
        return mine

    pipe = HybridPipeline(local_rank, rank=r_in if C > 1 else 0, world=C if C > 1 else 1, group=group_for(C))
    pipe.load_dense(wl.rows(lo, hi), id_base=lo)
    state = {"idx": None, "rerank": None}

    def need_bm25(p, c, lo_, hi_):
        from sentio_b200.index import build_bm25_from_token_ids

        if c > 1:   # every rank builds ITS doc range on its GPU; only (term, df) statistics are exchanged (all-gather)
            flat_l, off_l = wl.text_range(lo_, hi_)
            return p.build_bm25_sharded(flat_l, off_l, id_base=lo_, export=True)
        flat, off = wl.text()   # single shard: the index is built on the device (sb_bm25_build_*), 0.3 s at 1 M docs
        state["idx"] = p.engine.build_bm25_gpu(flat, off, export=True)
        return state["idx"]

    def need_rerank(p, c=1, lo_=0, hi_=None):
        from sentio_b200.cross_encoder import MINILM_L6, CrossEncoderWeights
        from sentio_b200.index import doc_token_matrix, hash_vocab_ids

        vocab_ids = hash_vocab_ids(wl.synth.VOCAB)
        if c > 1 and n > 2_000_000:
            # every rank tokenises its own doc range; the (small) uint16 token matrices are all-gathered over NCCL so any
            # global candidate can be framed locally (replicated: 240 B per doc)
            flat_l, off_l = wl.text_range(lo_, hi_)
            tok_l, len_l = doc_token_matrix(flat_l, off_l, vocab_ids, ld=120)
            per = (n + c - 1) // c
            tk = torch.zeros((per, tok_l.shape[1]), dtype=torch.int16, device=f"cuda:{local_rank}")
            ln = torch.zeros((per,), dtype=torch.int32, device=f"cuda:{local_rank}")
            tk[:len(tok_l)] = torch.from_numpy(tok_l.view(np.int16)).to(tk.device)
            ln[:len(len_l)] = torch.from_numpy(len_l.astype(np.int32)).to(ln.device)
            tk_all = torch.empty((c * per, tok_l.shape[1]), dtype=torch.int16, device=tk.device)
            ln_all = torch.empty((c * per,), dtype=torch.int32, device=tk.device)
            # (NCCL has no 16-bit integer type: the token matrix travels as bytes)
            dist.all_gather_into_tensor(tk_all.view(torch.uint8).view(-1), tk.view(torch.uint8).view(-1), group=group_for(c))
            dist.all_gather_into_tensor(ln_all, ln, group=group_for(c))
            bounds = [((n * r) // c, (n * (r + 1)) // c) for r in range(c)]
            doc_tok = np.concatenate([tk_all[r * per:r * per + (b_ - a_)].cpu().numpy().view(np.uint16)
                                      for r, (a_, b_) in enumerate(bounds)])
            doc_len = np.concatenate([ln_all[r * per:r * per + (b_ - a_)].cpu().numpy() for r, (a_, b_) in enumerate(bounds)])
        else:
            flat, off = wl.text()
            doc_tok, doc_len = doc_token_matrix(flat, off, vocab_ids, ld=120)
        p.load_cross_encoder(CrossEncoderWeights.random(MINILM_L6, seed=0))
        p.load_doc_tokens(doc_tok, doc_len, id_base=0)  # replicated on every rank (240 MB at 1 M docs)
        state["rerank"] = {"q_tok_all": vocab_ids[wl.q_tokens].astype(np.int32)}
        return state["rerank"]

    idx = need_bm25(pipe, C, lo, hi) if kind in ("hybrid", "rerank", "bm25") else None
    rr = need_rerank(pipe, C, lo, hi) if kind == "rerank" else None
    leg = Leg(kind, pipe, wl, args, world, rank, local_rank, C, my_group, lo, hi, idx, rr)
    res = leg.run(args.steps, args.warmup, capture=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, kind, res["outputs"])
    res["outputs"] = None
    roofline = leg.roofline_dense(res) if kind != "bm25" else {}
    if kind in ("hybrid", "rerank", "bm25"):
        roofline["bm25"] = leg.roofline_bm25(res)
    if kind == "rerank":
        roofline["cross_encoder"] = leg.roofline_ce(res)

    extras = set() if (args.no_extras or kind != "dense" or args.n_docs > 2_000_000) else set(args.extras.split(","))
    workloads, lat, part = {}, None, None
    sub_steps, sub_warm = args.steps, max(3, min(args.warmup, 3))

    def sub_leg(k2, p, c, lo_, hi_, my_group_, idx_, rr_):
        lg = Leg(k2, p, wl, args, world, rank, local_rank, c, my_group_, lo_, hi_, idx_, rr_)
        r = lg.run(sub_steps, sub_warm, sample_clocks=True)
        o = {"workload": workload_name(n, args.dim, k2, args.top_k, args.rerank_k), "value": r["value"], "unit": UNIT,
             "ms_per_step": r["ms_per_step"], "steps": sub_steps, "warmup": sub_warm, "queries_per_batch_per_gpu": lg.B_gpu,
             "batches_per_step": lg.inner, "timed_region_s": r["timed_region_s"], "e2e": r["e2e"],
             "gpu_launches": r["launches"], "clocks": r["clocks"], "roofline": {"dense_scan": lg.roofline_dense(r)}}
        if k2 in ("hybrid", "rerank"):
            o["roofline"]["bm25"] = lg.roofline_bm25(r)
        if k2 == "rerank":
            o["roofline"]["cross_encoder"] = lg.roofline_ce(r)
        return o, r

    if C == 1 and ("hybrid" in extras or "rerank" in extras or "latency_b1" in extras):
        idx = need_bm25(pipe, 1, 0, n)
    if C == 1 and "hybrid" in extras:
        workloads["hybrid"], _ = sub_leg("hybrid", pipe, 1, 0, n, my_group, idx, None)
    if C == 1 and "latency_b1" in extras and world == 1:
        lat = latency_b1(pipe, wl, idx)
    if C == 1 and "rerank" in extras:
        rr = need_rerank(pipe)
        workloads["rerank"], _ = sub_leg("rerank", pipe, 1, 0, n, my_group, idx, rr)

    # ---- north_star's multi-GPU layout on the SAME corpus: C = world corpus shards + one all-gather per batch
    if world > 1 and C == 1 and "partitioned" in extras:
        plo, phi = (n * rank) // world, (n * (rank + 1)) // world
        ppipe = HybridPipeline(local_rank, rank=rank, world=world, group=group_for(world))
        ppipe.load_dense(wl.rows(plo, phi), id_base=plo)
        ppipe.stage_timing = True
        pd, pr = sub_leg("dense", ppipe, world, plo, phi, 0, None, None)
        nb = pr["n_batches"]
        stage = {"sampling_passes+threshold_select_us": pr["prof"]["dense_sample"][1] / nb * 1e3,
                 "scan_us": pr["prof"]["dense_scan"][1] / nb * 1e3,
                 "window_select+fp64_rescore_us": pr["prof"]["dense_merge"][1] / nb * 1e3}
        stage.update({k_: v / max(ppipe.stage_counts.get(k_, 1), 1) * 1e3 for k_, v in ppipe.stage_ms().items()})
        part = {"layout": f"{world} corpus shards (contiguous doc ranges of the same {n}-doc corpus) x 1 query group; every "
                          f"rank scores the step's {world} x {pd['queries_per_batch_per_gpu']} queries against its shard, "
                          "ONE all_gather_into_tensor of the per-shard top-k records, merge_shards on global ranks",
                "dense": pd, "per_batch_stage_us_rank0": stage}
        if "hybrid" in extras:
            pidx = need_bm25(ppipe, world, plo, phi)
            ph, _ = sub_leg("hybrid", ppipe, world, plo, phi, 0, pidx, None)
            part["hybrid"] = ph
        ppipe.engine.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---------------- bounded CPU baselines on this box's host cores (rank 0, N=1 only)
    cpu = None
    if world == 1 and args.cpu_sample > 0 and args.n_docs <= 2_000_000:
        cpu, _ = cpu_reference(kind if kind != "bm25" else "dense", wl, args.cpu_sample, args.top_k, args.rerank_k)
        if "hybrid" in workloads:
            workloads["hybrid"]["cpu_baseline"], _ = cpu_reference("hybrid", wl, 8, args.top_k, args.rerank_k)
        if "rerank" in workloads:
            workloads["rerank"]["cpu_baseline"], _ = cpu_reference("rerank", wl, 2, args.top_k, args.rerank_k)
    if world == 1 and "bm25_10k" in extras:
        try:
            workloads["bm25_10k"] = bm25_10k_leg(local_rank)
        except Exception as exc:  # a broken extra leg must not cost the headline line
            workloads["bm25_10k"] = {"error": str(exc)}

    line = {"metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16 store / f32 scan / f64 exact re-score",
            "data": "synthetic", "config": config, "clocks": res["clocks"], "e2e": res["e2e"],
            "gpu_launches": res["launches"], "timed_region_s": res["timed_region_s"], "roofline": roofline,
            "cpu_baseline": cpu, "corpus_gen_s": round(wl.gen_s, 1)}
    if workloads:
        line["workloads"] = workloads
    if lat:
        line["latency_b1"] = lat
    if part:
        line["partitioned"] = part
    _emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
