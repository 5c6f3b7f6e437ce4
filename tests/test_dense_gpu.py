"""K1 parity: libsentio_b200 dense cosine top-k vs the exact fp64 oracle (ids + ranks identical, scores rel 1e-9)."""
import numpy as np
import pytest

from helpers import assert_topk_matches
from oracle import dense as dense_oracle

pytestmark = pytest.mark.gpu


def _check(engine, vecs, q, k, slot=0, id_base=0):
    engine.load_dense(vecs, id_base=id_base, slot=slot)
    rows16 = dense_oracle.stored_rows(vecs)
    ids, sc, cnt = engine.dense_topk(q, k, slot=slot)
    for b in range(len(q)):
        wi, ws = dense_oracle.dense_topk(rows16, q[b], k)
        assert_topk_matches(ids[b] - id_base, sc[b], cnt[b], wi, ws, what=f"n={len(vecs)} d={vecs.shape[1]} k={k} b={b}")
    return ids, sc, cnt


@pytest.mark.parametrize("n,d,k,B", [
    (1, 8, 5, 1), (7, 16, 10, 3), (31, 64, 10, 4), (33, 100, 7, 5), (1000, 768, 10, 2), (5000, 1024, 100, 7),
    (4096, 384, 100, 4), (3000, 1536, 50, 3), (2000, 2048, 10, 2), (600, 3072, 10, 2), (500, 4096, 20, 3),
    (20000, 256, 228, 2), (70000, 128, 100, 6), (150000, 64, 10, 1),
])
def test_dense_topk_matches_oracle_f16_corpus(engine, n, d, k, B):
    rng = np.random.default_rng(n * 31 + d)
    x = rng.standard_normal((n, d)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    q = rng.standard_normal((B, d)).astype(np.float32)
    _check(engine, x.astype(np.float16), q, k, id_base=1000)


@pytest.mark.parametrize("n,d,k,B", [(9000, 1024, 10, 16), (20000, 256, 100, 40), (30000, 768, 100, 70),
                                     (200000, 128, 228, 33), (12000, 64, 5, 130), (40000, 1024, 100, 260)])
def test_dense_batched_tcgen05_path_matches_oracle(engine, n, d, k, B):
    """B >= 16 queries take the tcgen05 batched-query scan (dense_mma.cu); results must equal the oracle AND be
    bit-identical to the CUDA-core scan."""
    rng = np.random.default_rng(n + d + B)
    x = rng.standard_normal((n, d)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    x16 = x.astype(np.float16)
    x16[100:140] = x16[50]          # a block of exact duplicates
    q = rng.standard_normal((B, d)).astype(np.float32)
    q[3] = x16[50].astype(np.float32)   # hits the duplicate block -> exact ties
    q[5] = 0.0                          # zero query -> all scores 0
    engine.dense_set_mode(0)
    ids, sc, cnt = _check(engine, x16, q, k, id_base=7)
    engine.dense_set_mode(1)
    ids1, sc1, cnt1 = engine.dense_topk(q, k)
    engine.dense_set_mode(0)
    assert np.array_equal(ids, ids1) and np.array_equal(sc, sc1) and np.array_equal(cnt, cnt1)


def test_dense_set_mode_accepts_only_auto_and_cuda_core(engine):
    from sentio_b200._lib import SentioB200Error

    for mode in (-1, 2):
        with pytest.raises(SentioB200Error):
            engine.dense_set_mode(mode)
    engine.dense_set_mode(1)
    engine.dense_set_mode(0)


def _near_tie_corpus(rng, n, d, cluster, ulps=1):
    """Random unit corpus whose rows [200, 200+cluster) are 1-ulp (fp16) perturbations of one base row: their cosines
    with any query differ by ~1e-6 .. 1e-5, far below the fp16-query rounding error of the tcgen05 scan."""
    x = rng.standard_normal((n, d)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    x16 = x.astype(np.float16)
    base = x16[7].copy()
    for j in range(cluster):
        row = base.copy()
        for c in rng.choice(d, size=1 + (j % 3), replace=False):
            row[c] = np.nextafter(row[c], np.float16(np.inf if (j + c) % 2 else -np.inf)) if ulps else row[c]
        x16[200 + j] = row
    return x16, base.astype(np.float32)


@pytest.mark.parametrize("n,d,k,B,cluster", [(20000, 256, 100, 16, 200), (40960, 1024, 100, 24, 200),
                                             (30000, 512, 10, 70, 64), (9000, 128, 50, 3, 120)])
def test_dense_near_tie_cluster_straddling_rank_k(engine, n, d, k, B, cluster):
    """VERDICT r01: a cluster of rows whose cosines differ by less than the approximate scores' error straddles rank k.
    The error-bounded hand-off window must re-score all of them: ids == oracle, for both scans."""
    rng = np.random.default_rng(n + cluster)
    x16, base = _near_tie_corpus(rng, n, d, cluster)
    q = rng.standard_normal((B, d)).astype(np.float32)
    q[0] = base                                      # the cluster is the top of the list, rank k falls inside it
    q[1] = base + 0.05 * rng.standard_normal(d).astype(np.float32)
    q[2] = 3.0 * base + 0.3 * rng.standard_normal(d).astype(np.float32)
    for mode in (0, 1):
        engine.dense_set_mode(mode)
        try:
            _check(engine, x16, q, k)
        finally:
            engine.dense_set_mode(0)


@pytest.mark.parametrize("B", [2, 20])
def test_dense_window_larger_than_the_winner_buffer_uses_the_exact_fallback(engine, B):
    """3000 near-identical rows on top: the window (> 2048 rows) cannot be re-scored in shared memory; the brute-force
    fp64 kernel must answer -- same ids as the oracle.  5000 EXACT duplicates exercise the tie order (lowest row first)."""
    rng = np.random.default_rng(77)
    x16, base = _near_tie_corpus(rng, 24000, 256, 3000)
    x16[8000:13000] = x16[9]                          # 5000 exact duplicates
    q = rng.standard_normal((B, 256)).astype(np.float32)
    q[0] = base
    q[1] = x16[9].astype(np.float32)
    ids, sc, cnt = _check(engine, x16, q, 10)
    assert list(ids[1]) == [9] + list(range(8000, 8009))


def test_dense_query_scale_does_not_change_the_result(engine):
    """ADVICE r01: cosine is scale invariant -- queries scaled by 1e6 / 1e-6 / 1e-30 / 1e30 must give the same ids on
    the CUDA-core scan (B = 1) and on the tcgen05 scan (B = 64), whose fp16 operand would otherwise overflow / vanish."""
    rng = np.random.default_rng(12)
    x = rng.standard_normal((20000, 256)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    engine.load_dense(x.astype(np.float16))
    q = rng.standard_normal((64, 256)).astype(np.float32)
    want, _, _ = engine.dense_topk(q, 50)
    for scale in (1e6, 1e-6, 1e30, 1e-30):
        qs = (q.astype(np.float64) * scale).astype(np.float32)
        got, sc, _ = engine.dense_topk(qs, 50)
        assert np.array_equal(got, want), f"batched, scale {scale}"
        one, sc1, _ = engine.dense_topk(qs[:1], 50)
        assert np.array_equal(one[0], want[0]), f"single, scale {scale}"
        assert np.all(np.isfinite(sc)) and np.all(np.abs(sc) <= 1.0 + 1e-9)


def test_dense_top_k_up_to_1024(engine):
    rng = np.random.default_rng(4)
    x = rng.standard_normal((30000, 128)).astype(np.float16)
    q = rng.standard_normal((18, 128)).astype(np.float32)
    _check(engine, x, q[:2], 1024)
    _check(engine, x, q, 1000)


def test_dense_f32_input_is_normalised_then_rounded(engine):
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((3000, 200)) * rng.uniform(0.1, 50, size=(3000, 1))).astype(np.float32)
    q = rng.standard_normal((3, 200)).astype(np.float32) * 7
    _check(engine, x, q, 25)
    stored = engine.dense_fetch(np.arange(10))
    assert np.array_equal(stored.astype(np.float16), dense_oracle.stored_rows(x)[:10])


def test_dense_ties_duplicates_and_zero_rows(engine):
    rng = np.random.default_rng(9)
    base = rng.standard_normal((50, 96)).astype(np.float32)
    x = np.concatenate([base] * 8 + [np.zeros((20, 96), np.float32)])  # every row appears 8 times + zero rows
    x16 = (x / np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-30)).astype(np.float16)
    q = base[:4] + 0.01
    ids, sc, cnt = _check(engine, x16, q, 20)
    # exact duplicates tie exactly: lowest index first
    for b in range(4):
        assert list(ids[b, :8]) == [b + 50 * j for j in range(8)]
    # zero query -> every score is 0 -> ids 0..k-1
    ids, sc, cnt = engine.dense_topk(np.zeros((1, 96), np.float32), 5)
    assert list(ids[0]) == [0, 1, 2, 3, 4] and np.all(sc == 0.0)


def test_dense_k_larger_than_corpus_and_empty_index(engine):
    rng = np.random.default_rng(2)
    x = rng.standard_normal((12, 32)).astype(np.float16)
    q = rng.standard_normal((2, 32)).astype(np.float32)
    ids, sc, cnt = _check(engine, x, q, 40)
    assert list(cnt) == [12, 12] and np.all(ids[:, 12:] == -1)
    engine.load_dense(np.zeros((0, 32), np.float16), slot=1)
    ids, sc, cnt = engine.dense_topk(q, 3, slot=1)
    assert list(cnt) == [0, 0]


def test_dense_device_entry_point_equals_host_entry_point(engine):
    import torch

    rng = np.random.default_rng(3)
    x = rng.standard_normal((9000, 512)).astype(np.float16)
    q = rng.standard_normal((9, 512)).astype(np.float32)
    engine.load_dense(x)
    h_ids, h_sc, h_cnt = engine.dense_topk(q, 64)
    d_ids, d_sc, d_cnt = engine.dense_topk_dev(torch.from_numpy(q).cuda(), 64)
    torch.cuda.synchronize()
    assert np.array_equal(d_ids.cpu().numpy(), h_ids) and np.array_equal(d_sc.cpu().numpy(), h_sc)
    assert np.array_equal(d_cnt.cpu().numpy(), h_cnt)


def test_dense_full_size_1m_x_1024(engine):
    """BASELINE config 2 shape: 1 M x 1024, top_k=100.  Oracle on 2 queries + size-independent properties."""
    from sentio_b200 import synth

    n, d, k = 1_000_000, 1024, 100
    x16 = synth.dense_corpus(n, d)
    q = synth.query_vectors(6, d)
    engine.load_dense(x16)
    # (a) self-retrieval: a stored row used as query must come back first with cosine 1
    probe = np.array([0, 123_456, 999_999])
    qs = np.concatenate([q, x16[probe].astype(np.float32)])
    ids, sc, cnt = engine.dense_topk(qs, k)
    assert list(ids[6:, 0]) == list(probe) and np.allclose(sc[6:, 0], 1.0, atol=1e-12)
    assert np.all(cnt == k)
    # (b) sortedness + uniqueness + every reported score is the exact cosine of that row
    for b in range(len(qs)):
        assert np.all(np.diff(sc[b]) <= 0) and len(set(ids[b])) == k
        exact = dense_oracle.cosine_scores(x16[ids[b]], qs[b])
        assert np.allclose(exact, sc[b], rtol=1e-9, atol=1e-12)
    # (c) linearity of the ranking: scaling the query does not change ids
    ids2, _, _ = engine.dense_topk(q[:2] * 3.5, k)
    assert np.array_equal(ids2, ids[:2])
    # (d) full oracle comparison on two queries
    for b in range(2):
        wi, ws = dense_oracle.dense_topk(x16, q[b], k)
        assert_topk_matches(ids[b], sc[b], cnt[b], wi, ws, what=f"1M b={b}")
    # (e) the bench configuration: a 256-query batch (two 128-query groups on the cta_group::2 pair kernel), compared
    #     with the oracle on 8 sampled queries and bit for bit with the CUDA-core scan on the first 64
    q256 = np.concatenate([synth.query_vectors(253, d, seed=99), x16[probe].astype(np.float32)])
    engine.dense_set_mode(0)
    a = engine.dense_topk(q256, k)
    picks = [0, 63, 64, 127, 128, 200, 252, 255]
    for b, (wi, ws) in zip(picks, dense_oracle.dense_topk_multi(x16, q256[picks], k)):
        assert_topk_matches(a[0][b], a[1][b], a[2][b], wi, ws, what=f"1M batch-256 b={b}")
    engine.dense_set_mode(1)
    b_ = engine.dense_topk(q256[:64], k)
    engine.dense_set_mode(0)
    assert np.array_equal(a[0][:64], b_[0]) and np.array_equal(a[1][:64], b_[1]) and np.array_equal(a[2][:64], b_[2])
    assert list(a[0][253:, 0]) == list(probe)
