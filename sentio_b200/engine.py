"""B200Engine -- thin Python owner of one ``sb_ctx`` (one GPU / one corpus shard).

Host-buffer methods take / return NumPy arrays and go through the host entry points of the C ABI (H2D/D2H inside the
call).  ``*_dev`` methods take / return torch CUDA tensors, enqueue on torch's CURRENT stream and do not synchronise;
they are what the batched hybrid path, the multi-GPU shard path and bench.py's device-resident leg use.
torch is plumbing here (device memory, streams, torch.distributed) -- all arithmetic runs in libsentio_b200.so.
"""
from __future__ import annotations

import ctypes as C
from typing import Sequence

import numpy as np

from ._lib import SbCeConfig, SentioB200Error, check, load_library
from .index import Bm25IndexData

FUSION_METHODS = {"rrf": 0, "weighted_rrf": 1, "comb_sum": 2}


def _ptr(a):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


def _tptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class B200Engine:
    def __init__(self, device: int = 0):
        self._lib = load_library()
        h = C.c_void_p()
        check(self._lib.sb_create(int(device), C.byref(h)), "sb_create")
        self._h = h
        self.device = int(device)
        self.dense_dim = {}
        self.dense_count = {}
        self.bm25: Bm25IndexData | None = None
        self.bm25_id_base = 0
        self.ce_config = None
        self._pinned: list = []

    # ------------------------------------------------------------------ lifetime
    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.sb_destroy(self._h)
            self._h = None
            for p in getattr(self, "_pinned", []):
                self._lib.sb_host_free(C.c_void_p(p))
            self._pinned = []

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @property
    def num_sms(self) -> int:
        return int(self._lib.sb_num_sms(self._h))

    def sync(self) -> None:
        check(self._lib.sb_sync(self._h), "sb_sync")

    def launch_count(self) -> int:
        return int(self._lib.sb_launch_count(self._h))

    PROF_IDS = {"dense_scan": 0, "dense_merge": 1, "bm25_score": 2, "bm25_select": 3, "fuse": 4, "ce": 5, "dense_sample": 6}

    def profile(self, enable: bool) -> None:
        check(self._lib.sb_profile(self._h, 1 if enable else 0), "sb_profile")

    def profile_read(self, kernel: str):
        n, ms = C.c_int64(0), C.c_double(0.0)
        check(self._lib.sb_profile_read(self._h, self.PROF_IDS[kernel], C.byref(n), C.byref(ms)), "sb_profile_read")
        return int(n.value), float(ms.value)

    def _stream(self):
        import torch

        # torch's default stream has handle 0, which the C ABI reserves for "the context's own stream": pass the
        # explicit legacy-default-stream handle (cudaStreamLegacy == 0x1) so our kernels stay ordered with torch ops
        h = torch.cuda.current_stream(self.device).cuda_stream
        return C.c_void_p(h if h else 1)

    # ------------------------------------------------------------------ K1 dense
    def load_dense(self, vecs: np.ndarray, id_base: int = 0, slot: int = 0) -> None:
        v = np.ascontiguousarray(vecs)
        if v.ndim != 2:
            raise ValueError("vecs must be [n, d]")
        if v.dtype == np.float16:
            dt = 1
        else:
            v = np.ascontiguousarray(v, dtype=np.float32)
            dt = 0
        n, d = v.shape
        check(self._lib.sb_dense_load(self._h, slot, _ptr(v), n, d, dt, int(id_base)), "sb_dense_load")
        self.dense_dim[slot] = d
        self.dense_count[slot] = n

    def dense_set_mode(self, mode: int) -> None:
        """0 = auto (batches of >= 16 queries use the tcgen05 batched scan when eligible), 1 = CUDA-core scan only."""
        check(self._lib.sb_dense_set_mode(self._h, int(mode)), "sb_dense_set_mode")

    def pinned_empty(self, shape, dtype) -> np.ndarray:
        """A page-locked NumPy array (``sb_host_alloc``): host entry points copy straight from / into such arrays, with
        no staging memcpy.  For callers that reuse their request / response buffers; freed with the engine."""
        shape = tuple(int(x) for x in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        dt = np.dtype(dtype)
        nbytes = max(1, int(np.prod(shape)) * dt.itemsize)
        p = self._lib.sb_host_alloc(nbytes)
        if not p:
            raise SentioB200Error("sb_host_alloc failed")
        self._pinned.append(p)
        buf = (C.c_uint8 * nbytes).from_address(p)
        return np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)

    def dense_topk(self, q: np.ndarray, k: int, slot: int = 0, out=None):
        """``out`` = (ids [B,k] int64, scores [B,k] float64, counts [B] int32) to be filled in place (e.g. page-locked
        arrays from ``pinned_empty``); fresh arrays otherwise."""
        q = np.ascontiguousarray(np.atleast_2d(q), dtype=np.float32)
        B, d = q.shape
        if slot not in self.dense_dim:
            raise SentioB200Error(f"dense slot {slot} has no index loaded")
        if d != self.dense_dim[slot]:
            raise ValueError(f"query dimension {d} != index dimension {self.dense_dim[slot]}")
        if out is None:
            out = (np.empty((B, k), dtype=np.int64), np.empty((B, k), dtype=np.float64), np.empty(B, dtype=np.int32))
        ids, sc, cnt = out
        if ids.shape != (B, k) or sc.shape != (B, k) or cnt.shape != (B,) or ids.dtype != np.int64 \
                or sc.dtype != np.float64 or cnt.dtype != np.int32 or not (ids.flags.c_contiguous and sc.flags.c_contiguous):
            raise ValueError("dense_topk: out must be (int64 [B,k], float64 [B,k], int32 [B]) C-contiguous arrays")
        check(self._lib.sb_dense_topk(self._h, slot, _ptr(q), B, k, _ptr(ids), _ptr(sc), _ptr(cnt)), "sb_dense_topk")
        return ids, sc, cnt

    def dense_topk_dev(self, q_t, k: int, slot: int = 0, out=None):
        import torch

        B, d = q_t.shape
        assert q_t.is_cuda and q_t.dtype == torch.float32 and q_t.is_contiguous()
        if out is None:
            dev = q_t.device
            out = (torch.empty((B, k), dtype=torch.int64, device=dev), torch.empty((B, k), dtype=torch.float64, device=dev),
                   torch.empty((B,), dtype=torch.int32, device=dev))
        ids, sc, cnt = out
        check(self._lib.sb_dense_topk_dev(self._h, slot, _tptr(q_t), B, k, _tptr(ids), _tptr(sc), _tptr(cnt),
                                          self._stream()), "sb_dense_topk_dev")
        return ids, sc, cnt

    def dense_fetch(self, ids: Sequence[int], slot: int = 0) -> np.ndarray:
        ids = np.ascontiguousarray(ids, dtype=np.int64)
        out = np.empty((len(ids), self.dense_dim[slot]), dtype=np.float32)
        check(self._lib.sb_dense_fetch(self._h, slot, _ptr(ids), len(ids), _ptr(out)), "sb_dense_fetch")
        return out

    # ------------------------------------------------------------------ K2 BM25
    def load_bm25(self, data: Bm25IndexData, id_base: int = 0) -> None:
        variant = 1 if data.variant == "plus" else 0
        indptr = np.ascontiguousarray(data.indptr, dtype=np.int64)
        post_doc = np.ascontiguousarray(data.post_doc, dtype=np.int32)
        post_tf = np.ascontiguousarray(data.post_tf, dtype=np.uint16)
        doc_len = np.ascontiguousarray(data.doc_len, dtype=np.int32)
        idf = np.ascontiguousarray(data.idf, dtype=np.float64)
        check(self._lib.sb_bm25_load(self._h, _ptr(indptr), _ptr(post_doc), _ptr(post_tf), len(idf), len(post_doc),
                                     _ptr(doc_len), len(doc_len), float(data.avgdl), _ptr(idf), variant, float(data.k1),
                                     float(data.b), float(data.delta), int(id_base)), "sb_bm25_load")
        self.bm25 = data
        self.bm25_id_base = int(id_base)

    def build_bm25_gpu(self, flat_tokens: np.ndarray, doc_offsets: np.ndarray, variant: str = "okapi", k1: float = 1.5,
                       b: float = 0.75, epsilon: float = 0.25, delta: float = 1.0, id_base: int = 0,
                       export: bool = False, stats_hook=None) -> Bm25IndexData:
        """Index build on the device (sb_bm25_build_*): sort-based CSR construction from an integer token stream, idf on
        the host from the device-computed df, index installed without the postings ever visiting the host
        (``export=True`` additionally copies the CSR back, for ``save`` / ``shard``).  Same index as
        ``index.build_bm25_from_token_ids`` + ``load_bm25`` (tests/test_bm25_build_gpu.py).

        ``stats_hook(term_token, df, n_docs, n_tokens) -> (idf_of_token, average_idf, avgdl)`` turns the build into one
        SHARD of a partitioned corpus: the hook exchanges the per-shard statistics (HybridPipeline.build_bm25_sharded
        all-gathers them) and returns the corpus-global idf / avgdl that this shard's postings are scored with."""
        from .index import finish_gpu_built_index

        variant = variant.lower()
        flat = np.ascontiguousarray(flat_tokens, dtype=np.int32)
        off = np.ascontiguousarray(doc_offsets, dtype=np.int64)
        n_docs = len(off) - 1
        if n_docs <= 0 or len(flat) == 0:
            raise ValueError("empty corpus")
        nt, nnz = C.c_int64(0), C.c_int64(0)
        check(self._lib.sb_bm25_build_tokens(self._h, _ptr(flat), len(flat), _ptr(off), n_docs, C.byref(nt),
                                             C.byref(nnz)), "sb_bm25_build_tokens")
        V, nnz = int(nt.value), int(nnz.value)
        df = np.empty(V, dtype=np.int64)
        term_token = np.empty(V, dtype=np.int32)
        check(self._lib.sb_bm25_build_read(self._h, _ptr(df), _ptr(term_token)), "sb_bm25_build_read")
        csr = None
        if export:
            csr = (np.empty(V + 1, np.int64), np.empty(nnz, np.int32), np.empty(nnz, np.uint16), np.empty(n_docs, np.int32))
            check(self._lib.sb_bm25_build_export(self._h, *[_ptr(a) for a in csr]), "sb_bm25_build_export")
        gstats = stats_hook(term_token, df, n_docs, len(flat)) if stats_hook is not None else None
        data = finish_gpu_built_index(df, term_token, n_docs, len(flat), variant, k1, b, epsilon, delta, csr, gstats)
        idf = np.ascontiguousarray(data.idf, dtype=np.float64)
        check(self._lib.sb_bm25_build_finish(self._h, _ptr(idf), float(data.avgdl), 1 if variant == "plus" else 0,
                                             float(k1), float(b), float(delta), int(id_base)), "sb_bm25_build_finish")
        self.bm25 = data
        self.bm25_id_base = int(id_base)
        return data

    @staticmethod
    def pack_queries(term_id_lists: Sequence[Sequence[int]]):
        """-> (flat int32 term ids (at least one slot), CSR offsets int32 [B+1])"""
        lens = np.fromiter((len(t) for t in term_id_lists), dtype=np.int32, count=len(term_id_lists))
        off = np.zeros(len(term_id_lists) + 1, dtype=np.int32)
        np.cumsum(lens, out=off[1:])
        if int(off[-1]) == 0:
            return np.zeros(1, dtype=np.int32), off
        flat = np.concatenate([np.asarray(t, dtype=np.int32) for t in term_id_lists])
        return flat, off

    def bm25_topk(self, term_id_lists: Sequence[Sequence[int]], k: int):
        B = len(term_id_lists)
        flat, off = self.pack_queries(term_id_lists)
        ids = np.empty((B, k), dtype=np.int64)
        sc = np.empty((B, k), dtype=np.float64)
        cnt = np.empty(B, dtype=np.int32)
        check(self._lib.sb_bm25_topk(self._h, _ptr(flat), _ptr(off), B, k, _ptr(ids), _ptr(sc), _ptr(cnt)),
              "sb_bm25_topk")
        return ids, sc, cnt

    def bm25_topk_dev(self, terms_t, off_t, B: int, n_terms: int, max_len: int, k: int, out=None):
        import torch

        if out is None:
            dev = off_t.device
            out = (torch.empty((B, k), dtype=torch.int64, device=dev), torch.empty((B, k), dtype=torch.float64, device=dev),
                   torch.empty((B,), dtype=torch.int32, device=dev))
        ids, sc, cnt = out
        check(self._lib.sb_bm25_topk_dev(self._h, _tptr(terms_t), _tptr(off_t), B, n_terms, max_len, k, _tptr(ids),
                                         _tptr(sc), _tptr(cnt), self._stream()), "sb_bm25_topk_dev")
        return ids, sc, cnt

    def bm25_scores(self, term_ids: Sequence[int]) -> np.ndarray:
        t = np.ascontiguousarray(term_ids, dtype=np.int32)
        n = int(self._lib.sb_bm25_count(self._h))
        out = np.zeros(n, dtype=np.float64)
        check(self._lib.sb_bm25_scores(self._h, _ptr(t), len(t), _ptr(out)), "sb_bm25_scores")
        return out

    # ------------------------------------------------------------------ K3 fusion
    def fuse(self, method: str, rrf_k: float, w_dense: float, w_sparse: float, k: int, dense=None, sparse=None,
             plugin=None, extra: np.ndarray | None = None):
        """Each list is (ids [B,stride] int64, scores [B,stride] float64, counts [B] int32) or None.

        ``extra``: [B, n_extra, e_stride] float64 or None.  Returns (ids, scores, src, counts)."""
        if method not in FUSION_METHODS:
            raise ValueError(f"Unknown fusion_method: {method}")  # same error the reference raises (hybrid.py:238)
        lists = []
        B = None
        for lst in (dense, sparse, plugin):
            if lst is None:
                lists.append((None, None, None, 0))
                continue
            i = np.ascontiguousarray(np.atleast_2d(lst[0]), dtype=np.int64)
            s = np.ascontiguousarray(np.atleast_2d(lst[1]), dtype=np.float64)
            c = np.ascontiguousarray(np.atleast_1d(lst[2]), dtype=np.int32)
            B = i.shape[0] if B is None else B
            assert i.shape == s.shape and i.shape[0] == B and c.shape[0] == B
            lists.append((i, s, c, i.shape[1]))
        if B is None:
            raise ValueError("fuse needs at least one list")
        n_extra = e_stride = 0
        ex = None
        if extra is not None and extra.size:
            ex = np.ascontiguousarray(extra, dtype=np.float64)
            assert ex.ndim == 3 and ex.shape[0] == B
            n_extra, e_stride = ex.shape[1], ex.shape[2]
        ids = np.empty((B, k), dtype=np.int64)
        sc = np.empty((B, k), dtype=np.float64)
        src = np.empty((B, k), dtype=np.int32)
        cnt = np.empty(B, dtype=np.int32)
        (di, ds, dn, dstr), (si, ss, sn, sstr), (pi, ps, pn, pstr) = lists
        check(self._lib.sb_fuse(self._h, FUSION_METHODS[method], float(rrf_k), float(w_dense), float(w_sparse), B,
                                _ptr(di), _ptr(ds), _ptr(dn), dstr, _ptr(si), _ptr(ss), _ptr(sn), sstr,
                                _ptr(pi), _ptr(ps), _ptr(pn), pstr, _ptr(ex), n_extra, e_stride, k,
                                _ptr(ids), _ptr(sc), _ptr(src), _ptr(cnt)), "sb_fuse")
        return ids, sc, src, cnt

    def fuse_dev(self, method: str, rrf_k: float, w_dense: float, w_sparse: float, k: int, dense, sparse, out=None):
        import torch

        di, ds, dn = dense
        si, ss, sn = sparse
        B = di.shape[0]
        if out is None:
            dev = di.device
            out = (torch.empty((B, k), dtype=torch.int64, device=dev), torch.empty((B, k), dtype=torch.float64, device=dev),
                   torch.empty((B, k), dtype=torch.int32, device=dev), torch.empty((B,), dtype=torch.int32, device=dev))
        ids, sc, src, cnt = out
        check(self._lib.sb_fuse_dev(self._h, FUSION_METHODS[method], float(rrf_k), float(w_dense), float(w_sparse), B,
                                    _tptr(di), _tptr(ds), _tptr(dn), di.shape[1], _tptr(si), _tptr(ss), _tptr(sn),
                                    si.shape[1], None, None, None, 0, None, 0, 0, k, _tptr(ids), _tptr(sc), _tptr(src),
                                    _tptr(cnt), self._stream()), "sb_fuse_dev")
        return ids, sc, src, cnt

    def hybrid_topk(self, q: np.ndarray, flat_terms: np.ndarray, off: np.ndarray, k: int, method: str = "rrf",
                    rrf_k: float = 60, w_dense: float = 0.5, w_sparse: float = 0.5):
        """Whole retrieve -> fuse path from host buffers (sb_hybrid_topk): (ids, scores, src, counts) NumPy arrays."""
        q = np.ascontiguousarray(q, dtype=np.float32)
        flat = np.ascontiguousarray(flat_terms, dtype=np.int32)
        off = np.ascontiguousarray(off, dtype=np.int32)
        B = q.shape[0]
        ids = np.empty((B, k), dtype=np.int64)
        sc = np.empty((B, k), dtype=np.float64)
        src = np.empty((B, k), dtype=np.int32)
        cnt = np.empty(B, dtype=np.int32)
        check(self._lib.sb_hybrid_topk(self._h, _ptr(q), _ptr(flat), _ptr(off), B, int(k), FUSION_METHODS[method],
                                       float(rrf_k), float(w_dense), float(w_sparse), _ptr(ids), _ptr(sc), _ptr(src),
                                       _ptr(cnt)), "sb_hybrid_topk")
        return ids, sc, src, cnt

    def hybrid_rerank_topk(self, q: np.ndarray, flat_terms: np.ndarray, off: np.ndarray, q_tok: np.ndarray,
                           q_len: np.ndarray, k: int, k_out: int, seq_len: int = 128, method: str = "rrf",
                           rrf_k: float = 60, w_dense: float = 0.5, w_sparse: float = 0.5):
        """retrieve -> fuse -> rerank from host buffers (sb_hybrid_rerank_topk): (ids, sigmoid scores, counts)."""
        q = np.ascontiguousarray(q, dtype=np.float32)
        flat = np.ascontiguousarray(flat_terms, dtype=np.int32)
        off = np.ascontiguousarray(off, dtype=np.int32)
        qt = np.ascontiguousarray(q_tok, dtype=np.int32)
        ql = np.ascontiguousarray(q_len, dtype=np.int32)
        B = q.shape[0]
        ids = np.empty((B, k_out), dtype=np.int64)
        sc = np.empty((B, k_out), dtype=np.float32)
        cnt = np.empty(B, dtype=np.int32)
        check(self._lib.sb_hybrid_rerank_topk(self._h, _ptr(q), _ptr(flat), _ptr(off), _ptr(qt), _ptr(ql), qt.shape[1], B,
                                              int(k), int(k_out), int(seq_len), FUSION_METHODS[method], float(rrf_k),
                                              float(w_dense), float(w_sparse), _ptr(ids), _ptr(sc), _ptr(cnt)),
              "sb_hybrid_rerank_topk")
        return ids, sc, cnt

    # ------------------------------------------------------------------ K4 scorers
    def semantic_mmr(self, q: np.ndarray, cand: np.ndarray | None = None, cand_ids=None, w_sem: float = 0.7,
                     lambda_: float = 0.7, w_mmr: float = 0.5, want_sem: bool = True, want_mmr: bool = True,
                     slot: int = 0):
        q = np.ascontiguousarray(q, dtype=np.float32).reshape(-1)
        d = q.shape[0]
        if cand is not None:
            cand = np.ascontiguousarray(cand, dtype=np.float32)
            n = cand.shape[0]
            assert cand.ndim == 2 and cand.shape[1] == d
            ids = None
        else:
            ids = np.ascontiguousarray(cand_ids, dtype=np.int64)
            n = len(ids)
        sem = np.zeros(n, dtype=np.float64) if want_sem else None
        mmr = np.zeros(n, dtype=np.float64) if want_mmr else None
        if n:
            check(self._lib.sb_semantic_mmr(self._h, slot, _ptr(q), d, _ptr(cand), _ptr(ids), n, float(w_sem),
                                            float(lambda_), float(w_mmr), _ptr(sem), _ptr(mmr)), "sb_semantic_mmr")
        return sem, mmr

    # ------------------------------------------------------------------ K5 cross-encoder
    def ce_load(self, weights: np.ndarray, cfg: dict) -> None:
        w = np.ascontiguousarray(weights, dtype=np.float32).reshape(-1)
        c = SbCeConfig(int(cfg["vocab_size"]), int(cfg["hidden"]), int(cfg["layers"]), int(cfg["heads"]),
                       int(cfg["intermediate"]), int(cfg["max_pos"]), int(cfg.get("type_vocab", 2)),
                       float(cfg.get("ln_eps", 1e-12)))
        check(self._lib.sb_ce_load(self._h, _ptr(w), w.size, C.byref(c)), "sb_ce_load")
        self.ce_config = dict(cfg)

    def enc_load(self, weights: np.ndarray, cfg: dict, proj_w: np.ndarray | None = None,
                 proj_b: np.ndarray | None = None) -> None:
        """Load the on-device embedder (sb_enc_load): encoder blob + optional [out_dim, hidden] output projection."""
        w = np.ascontiguousarray(weights, dtype=np.float32).reshape(-1)
        c = SbCeConfig(int(cfg["vocab_size"]), int(cfg["hidden"]), int(cfg["layers"]), int(cfg["heads"]),
                       int(cfg["intermediate"]), int(cfg["max_pos"]), int(cfg.get("type_vocab", 2)),
                       float(cfg.get("ln_eps", 1e-12)))
        pw = pb = None
        out_dim = 0
        if proj_w is not None:
            pw = np.ascontiguousarray(proj_w, dtype=np.float32)
            pb = np.ascontiguousarray(proj_b, dtype=np.float32)
            out_dim = int(pw.shape[0])
            if pw.shape != (out_dim, int(cfg["hidden"])) or pb.shape != (out_dim,):
                raise ValueError("proj_w must be [out_dim, hidden] and proj_b [out_dim]")
        check(self._lib.sb_enc_load(self._h, _ptr(w), w.size, C.byref(c), _ptr(pw), _ptr(pb), out_dim), "sb_enc_load")
        self.enc_config = dict(cfg)

    def enc_dim(self) -> int:
        return int(self._lib.sb_enc_dim(self._h))

    def enc_embed(self, input_ids: np.ndarray, token_type: np.ndarray, lengths: np.ndarray, normalize: bool = True):
        ids = np.ascontiguousarray(input_ids, dtype=np.int32)
        tt = np.ascontiguousarray(token_type, dtype=np.int32)
        ln = np.ascontiguousarray(lengths, dtype=np.int32)
        P, S = ids.shape
        out = np.empty((P, self.enc_dim()), dtype=np.float32)
        check(self._lib.sb_enc_embed(self._h, _ptr(ids), _ptr(tt), _ptr(ln), P, S, int(normalize), _ptr(out)),
              "sb_enc_embed")
        return out

    def enc_embed_dev(self, ids_t, tt_t, len_t, normalize: bool = True, out=None):
        import torch

        P, S = ids_t.shape
        if out is None:
            out = torch.empty((P, self.enc_dim()), dtype=torch.float32, device=ids_t.device)
        check(self._lib.sb_enc_embed_dev(self._h, _tptr(ids_t), _tptr(tt_t), _tptr(len_t), P, S, int(normalize),
                                         _tptr(out), self._stream()), "sb_enc_embed_dev")
        return out

    def ce_tokens_load(self, doc_tok: np.ndarray, doc_len: np.ndarray, id_base: int = 0) -> None:
        t = np.ascontiguousarray(doc_tok, dtype=np.uint16)
        ln = np.ascontiguousarray(doc_len, dtype=np.int32)
        check(self._lib.sb_ce_tokens_load(self._h, _ptr(t), _ptr(ln), t.shape[0], t.shape[1], int(id_base)),
              "sb_ce_tokens_load")

    def rerank_dev(self, q_tok_t, q_len_t, cand_ids_t, cand_cnt_t, S: int, k_out: int, out=None):
        import torch

        B, k = cand_ids_t.shape
        if out is None:
            dev = cand_ids_t.device
            out = (torch.empty((B, k_out), dtype=torch.int64, device=dev),
                   torch.empty((B, k_out), dtype=torch.float32, device=dev),
                   torch.empty((B,), dtype=torch.int32, device=dev))
        check(self._lib.sb_rerank_dev(self._h, _tptr(q_tok_t), _tptr(q_len_t), q_tok_t.shape[1], _tptr(cand_ids_t),
                                      _tptr(cand_cnt_t), B, k, int(S), int(k_out), _tptr(out[0]), _tptr(out[1]),
                                      _tptr(out[2]), self._stream()), "sb_rerank_dev")
        return out

    def load_doc_chars(self, n_chars: np.ndarray, id_base: int = 0) -> None:
        """K7 input: characters of every document's usable text (0 = blank); see sentio_b200.selector.selector_chars."""
        a = np.ascontiguousarray(n_chars, dtype=np.int32)
        check(self._lib.sb_doc_chars_load(self._h, _ptr(a), len(a), int(id_base)), "sb_doc_chars_load")

    def select_dev(self, cand_ids_t, cand_scores_t, cand_cnt_t, top_k: int, max_tokens: int, out=None):
        """Batched document selector (sb_select_dev) on device tensors; scores float32 or float64."""
        import torch

        B, k = cand_ids_t.shape
        dt = {torch.float32: 0, torch.float64: 1}[cand_scores_t.dtype]
        if out is None:
            dev = cand_ids_t.device
            out = (torch.empty((B, top_k), dtype=torch.int64, device=dev),
                   torch.empty((B, top_k), dtype=cand_scores_t.dtype, device=dev),
                   torch.empty((B,), dtype=torch.int32, device=dev), torch.empty((B,), dtype=torch.int32, device=dev))
        check(self._lib.sb_select_dev(self._h, _tptr(cand_ids_t), _tptr(cand_scores_t), dt, _tptr(cand_cnt_t), B, k,
                                      int(top_k), int(max_tokens), _tptr(out[0]), _tptr(out[1]), _tptr(out[2]),
                                      _tptr(out[3]), self._stream()), "sb_select_dev")
        return out

    def ce_gemm_test(self, a: np.ndarray, w: np.ndarray, bias: np.ndarray, epi: int, residual: np.ndarray | None = None):
        a = np.ascontiguousarray(a, dtype=np.float32)
        w = np.ascontiguousarray(w, dtype=np.float32)
        bias = np.ascontiguousarray(bias, dtype=np.float32)
        M, K = a.shape
        N = w.shape[0]
        res = None if residual is None else np.ascontiguousarray(residual, dtype=np.float32)
        out = np.empty((M, N), dtype=np.float32)
        check(self._lib.sb_ce_gemm_test(self._h, _ptr(a), _ptr(w), _ptr(bias), _ptr(res), M, N, K, int(epi), _ptr(out)),
              "sb_ce_gemm_test")
        return out

    def ce_score(self, input_ids: np.ndarray, token_type: np.ndarray, lengths: np.ndarray):
        ids = np.ascontiguousarray(input_ids, dtype=np.int32)
        tt = np.ascontiguousarray(token_type, dtype=np.int32)
        ln = np.ascontiguousarray(lengths, dtype=np.int32)
        P, S = ids.shape
        logits = np.empty(P, dtype=np.float32)
        sig = np.empty(P, dtype=np.float32)
        if P:
            check(self._lib.sb_ce_score(self._h, _ptr(ids), _ptr(tt), _ptr(ln), P, S, _ptr(logits), _ptr(sig)),
                  "sb_ce_score")
        return logits, sig

    def ce_stats(self, reset: bool = False):
        """(pairs, token rows computed, sum of squared pair lengths) of the packed-token forward since the last reset."""
        out = np.zeros(3, dtype=np.int64)
        check(self._lib.sb_ce_stats(self._h, _ptr(out), int(reset)), "sb_ce_stats")
        return int(out[0]), int(out[1]), int(out[2])

    def ce_score_dev(self, ids_t, tt_t, len_t, out=None):
        import torch

        P, S = ids_t.shape
        if out is None:
            out = (torch.empty((P,), dtype=torch.float32, device=ids_t.device),
                   torch.empty((P,), dtype=torch.float32, device=ids_t.device))
        check(self._lib.sb_ce_score_dev(self._h, _tptr(ids_t), _tptr(tt_t), _tptr(len_t), P, S, _tptr(out[0]),
                                        _tptr(out[1]), self._stream()), "sb_ce_score_dev")
        return out

    # ------------------------------------------------------------------ K6 shard merge
    def merge_shards_dev(self, ids0, scores0, counts0, shard_stride_bytes: int, G: int, out=None):
        """ids0/scores0/counts0: shard 0's [B,k] / [B,k] / [B] views inside the all-gathered record buffer."""
        import torch

        B, k = ids0.shape
        if out is None:
            dev = ids0.device
            out = (torch.empty((B, k), dtype=torch.int64, device=dev), torch.empty((B, k), dtype=torch.float64, device=dev),
                   torch.empty((B,), dtype=torch.int32, device=dev))
        check(self._lib.sb_merge_shards_dev(self._h, _tptr(ids0), _tptr(scores0), _tptr(counts0),
                                            int(shard_stride_bytes), int(G), B, k, _tptr(out[0]), _tptr(out[1]),
                                            _tptr(out[2]), self._stream()), "sb_merge_shards_dev")
        return out
