// bm25.cu -- K2: BM25 term-at-a-time scoring over term-major CSR postings + exact top-k.
//
// Replaces rank_bm25 0.2.2 BM25Okapi/BM25Plus.get_scores followed by np.argsort / `score > 0`
// (reference call sites src/core/retrievers/sparse.py:177-198).
//
// Bit-exactness contract (fp64, no FMA contraction -- every operation below is an explicit __d*_rn intrinsic):
//   dnorm[d]  = k1 * ((1 - b) + (b * dl[d]) / avgdl)                      (load time)
//   ratio[p]  = (tf[p] * (k1 + 1)) / (tf[p] + dnorm[doc[p]])              (load time, query independent)
//   Okapi:  score[d] += idf[t] * ratio[p]            for every posting p of query term t, terms in QUERY ORDER
//   Plus :  score[d] += idf[t] * (delta + ratio or 0.0)   for EVERY doc d (rank_bm25 adds delta to all docs)
// A doc occurs at most once in a term's posting list and the terms of a query are applied one after the other (block
// barrier in between), so no atomics are needed and the per-doc addition order equals NumPy's `score += ...` loop order.
//
// Algorithmic bytes per query: sum_t df(t) * (4 B doc + 8 B ratio): the accumulators of a doc range live in shared
// memory (bm25_range_kernel below), nothing of size N is ever written or re-read in HBM / L2 (DESIGN.md K2).
#include <algorithm>
#include <type_traits>
#include <string.h>
#include <utility>
#include <vector>

#include "common.cuh"

namespace {

// ------------------------------------------------------------------------------------------------ load kernels
__global__ void bm25_dnorm_kernel(const int32_t* __restrict__ doc_len, int64_t n, double k1, double b, double omb,
                                  double avgdl, double* __restrict__ dnorm) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double t1 = __dmul_rn(b, (double)doc_len[i]);
  const double t2 = __ddiv_rn(t1, avgdl);
  const double t4 = __dadd_rn(omb, t2);
  dnorm[i] = __dmul_rn(k1, t4);
}

__global__ void bm25_ratio_kernel(const int32_t* __restrict__ post_doc, const uint16_t* __restrict__ post_tf,
                                  int64_t nnz, const double* __restrict__ dnorm, double k1p1,
                                  double* __restrict__ ratio) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nnz) return;
  const double tf = (double)post_tf[i];
  const double num = __dmul_rn(tf, k1p1);
  const double den = __dadd_rn(tf, dnorm[post_doc[i]]);
  ratio[i] = __ddiv_rn(num, den);
}

// Dense rows of the head terms: one CTA per (slot, chunk of the term's posting list) scatters ratio[p] to row[doc[p]].
__global__ void bm25_dense_fill_kernel(const int64_t* __restrict__ indptr, const int32_t* __restrict__ post_doc,
                                       const double* __restrict__ ratio, const int32_t* __restrict__ slot_term,
                                       int64_t n_docs, double* __restrict__ dense) {
  const int slot = blockIdx.y;
  const int64_t lo = indptr[slot_term[slot]], hi = indptr[slot_term[slot] + 1];
  double* row = dense + (size_t)slot * n_docs;
  for (int64_t p = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < hi; p += (int64_t)gridDim.x * blockDim.x)
    row[post_doc[p]] = ratio[p];
}

// ------------------------------------------------------------------------------------------------ range scoring
// One CTA scores ONE query over a run of consecutive doc ranges of kRange docs.  The fp64 accumulators live in shared
// memory (64 KB per CTA), so the only memory traffic of scoring is the postings themselves (4 B doc + 8 B ratio each, most
// of them L2 hits: the head terms' lists are shared by the queries of a batch): no N x 8 B zero fill, no accumulator
// read-modify-write through L2, no N x 8 B re-read for the top-k.
//
// WARP-PRIVATE STRIPS (round 2; round 1 walked every (range, term) with the whole CTA and two block barriers per step --
// 69 thread instructions per posting, issue bound):
//  * the CTA's doc span is cut into 16 contiguous strips, one per warp; a warp walks its strip in sub-ranges of kSub = 512
//    docs whose accumulators are its private 4 KB slice of shared memory -- no block barrier after the set-up;
//  * postings of a term are sorted by doc, so a strip's slice of a posting list is contiguous: its start is found once
//    per (warp, term) with a warp-cooperative 32-ary search and then carried from sub-range to sub-range;
//  * inside a sub-range the terms are applied strictly in QUERY ORDER by the same warp (a doc occurs at most once per
//    posting list), so the per-doc addition order equals NumPy's `score += ...` loop order without any atomics
//    => bit-identical fp64 (every operation is an explicit __dmul_rn / __dadd_rn);
//  * HEAD TERMS (df >= n_docs / 4; a handful of stop-word-like terms carry ~90 % of all postings of a Zipf corpus) are
//    not walked through their posting lists at all: the index keeps a dense fp64 row ratio[doc] (0.0 = no posting) for each
//    of them and the warp adds idf * row[doc] to all 512 docs of the sub-range -- 16 independent, perfectly coalesced loads,
//    no cursor, no compare, no vote (8 instead of ~37 instructions per 32 postings).  Adding idf * 0.0 = +-0.0 to a doc
//    without a posting leaves its accumulator bit-for-bit unchanged, exactly like rank_bm25's dense `score +=` does;
//  * the posting-list walk addresses its shared-memory accumulators through 32-bit shared-space addresses and is
//    branch-free (a posting beyond the sub-range reads a never-written per-warp dummy slot): the first version spent
//    150 instructions per 128 postings on generic-address arithmetic and divergence bookkeeping (profiles/r02_run4_bm25*);
//  * a finished sub-range is consumed by its warp according to MODE:
//      kModeSample : (S ranges spread over the corpus, one per CTA) ceil(k/S)-th best positive score of the range, min
//                    over the S ranges -> thr[q], a lower bound of the global k-th best score
//      kModeCollect: every doc with score > 0 and >= thr[q] is appended to the query's candidate list
//      kModeDump   : the accumulators are written to out[q][doc] (sb_bm25_scores, the bit-exactness hook)
constexpr int kRange = 8192;            // docs per range (= 16 warps x kSub)
constexpr unsigned long long kPosZero = 0x8000000000000000ull;  // f64_orderable(+0.0)
constexpr int kRsThreads = 512;
constexpr int kRsWarps = kRsThreads / 32;
constexpr int kSub = kRange / kRsWarps; // docs per warp sub-range
constexpr int kRsPost = 4;              // 32-posting chunks a warp keeps in flight for the long lists
enum { kModeSample = 0, kModeCollect = 1, kModeDump = 2 };

struct RangeParams {
  const int32_t* q_terms;
  const int32_t* q_off;  // offsets of THIS sub-batch (q_off[0] may be > 0)
  int max_len;           // longest query of the sub-batch (sizes the per-term state in shared memory)
  int ranges_per_cta;
  const int64_t* indptr;
  const int32_t* post_doc;
  const double* ratio;
  const double* idf;
  const int32_t* dense_of_term;  // [V] slot of the term's dense ratio row, -1 = posting list only
  const double* dense_ratio;     // [n_dense][n_docs]
  int64_t n_terms;
  int64_t n_docs;
  double delta;          // BM25Plus
  int k;                 // kModeSample: rank inside one sample range = ceil(top_k / number of sample ranges)
  unsigned long long* thr;   // [nq]
  int32_t* cnt;              // [nq]
  unsigned long long* ckey;  // [nq][n_docs]   kModeCollect
  uint32_t* cidx;            // [nq][n_docs]
  double* dump;              // [nq][n_docs]   kModeDump
};

// first p in [lo, hi) with a[p] >= target (hi if none); all 32 lanes of the warp participate and return the same value
__device__ __forceinline__ int64_t warp_lower_bound(const int32_t* __restrict__ a, int64_t lo, int64_t hi, int32_t target,
                                                    int lane) {
  while (hi - lo > 32) {
    const int64_t step = (hi - lo + 31) / 32;  // >= 2
    const int64_t p = lo + (int64_t)lane * step;
    const bool ge = (p >= hi) || (__ldg(a + p) >= target);
    const unsigned m = __ballot_sync(0xffffffffu, ge);
    if (m == 0u) {
      lo = lo + 31 * step + 1;
    } else {
      const int f = __ffs(m) - 1;
      if (f == 0) {
        hi = lo;
      } else {
        hi = min(hi, lo + (int64_t)f * step);  // lane f may have probed past the end of the list
        lo = lo + (int64_t)(f - 1) * step + 1;
      }
    }
  }
  const int64_t p = lo + lane;
  const bool ge = (p >= hi) || (__ldg(a + p) >= target);
  const unsigned m = __ballot_sync(0xffffffffu, ge);
  return m ? lo + (__ffs(m) - 1) : hi;
}

__device__ unsigned long long block_kth_largest(const unsigned long long* keys, int n, int K, int* hist, int* scal,
                                                int passes);

__device__ __forceinline__ double lds_f64(uint32_t addr) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f64(uint32_t addr, double v) {
  asm volatile("st.shared.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}

template <int MODE, bool PLUS>
__global__ void __launch_bounds__(kRsThreads, 2) bm25_range_kernel(const RangeParams p) {
  extern __shared__ __align__(16) uint8_t rsm[];
  double* acc = reinterpret_cast<double*>(rsm);                               // [kRange]: warp w owns [w*kSub, (w+1)*kSub)
  double* s_dummy = acc + kRange;                                             // [kRsWarps] 0.0, read by out-of-range postings
  int64_t* s_lo = reinterpret_cast<int64_t*>(s_dummy + kRsWarps);             // [max_len] first posting of the term's list
  double* s_idf = reinterpret_cast<double*>(s_lo + p.max_len);                // [max_len] 0.0 = term contributes nothing
  int32_t* s_n = reinterpret_cast<int32_t*>(s_idf + p.max_len);               // [max_len] postings in the list (df < 2^31)
  int32_t* s_wid = s_n + p.max_len;                                           // [max_len] chunks in flight; -1 - slot = dense row
  int32_t* s_cur = s_wid + p.max_len;                                         // [kRsWarps][max_len] cursor, relative to s_lo
  uint32_t* s_bits = reinterpret_cast<uint32_t*>(s_cur + (size_t)kRsWarps * p.max_len);  // [kRange / 32] PLUS: doc had a posting
  __shared__ int hist[256];
  __shared__ int scal[4];
  __shared__ int npos;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int qi = blockIdx.x;
  const int64_t n_ranges = (p.n_docs + kRange - 1) / kRange;
  // kModeSample: gridDim.y sample ranges spread evenly over the corpus, one per CTA
  const int64_t first = MODE == kModeSample ? ((int64_t)blockIdx.y * n_ranges) / gridDim.y
                                            : (int64_t)blockIdx.y * p.ranges_per_cta;
  const int64_t last = MODE == kModeSample ? first + 1 : min(first + (int64_t)p.ranges_per_cta, n_ranges);  // exclusive
  const int q0 = p.q_off[qi];
  const int len = min(p.q_off[qi + 1] - q0, p.max_len);
  // per-term state shared by the CTA
  for (int j = tid; j < len; j += kRsThreads) {
    const int t = p.q_terms[q0 + j];
    double w = 0.0;
    int64_t lo = 0, hi = 0;
    int wid = 1;
    if (t >= 0 && t < p.n_terms) {
      w = p.idf[t];
      if (w != 0.0) {
        lo = p.indptr[t];
        hi = p.indptr[t + 1];
        const int slot = p.dense_of_term ? p.dense_of_term[t] : -1;
        // expected postings of the term inside one sub-range -> chunks kept in flight (rare terms must not over-read)
        const int64_t per_sub = ((hi - lo) * kSub) / max(p.n_docs, (int64_t)1);
        wid = slot >= 0 ? -1 - slot : (per_sub < 48 ? 1 : kRsPost);
      }
    }
    s_lo[j] = lo;
    s_n[j] = (int32_t)(hi - lo);
    s_idf[j] = w;
    s_wid[j] = wid;
  }
  double* a = acc + warp * kSub;
  const uint32_t a_s = smem_u32(a);                      // shared-space address of this warp's accumulators
  const uint32_t dummy_s = smem_u32(s_dummy + warp);
  for (int i = lane; i < kSub; i += 32) a[i] = 0.0;
  if (lane == 0) s_dummy[warp] = 0.0;
  uint32_t* bits = s_bits + warp * (kSub / 32);
  if (PLUS && lane < kSub / 32) bits[lane] = 0u;
  __syncthreads();

  // this warp's strip: kSub * (ranges of the CTA) consecutive docs
  const int64_t strip_len = (last - first) * kSub;
  const int64_t strip0 = first * kRange + (int64_t)warp * strip_len;
  int32_t* my_cur = s_cur + (size_t)warp * p.max_len;
  for (int j = 0; j < len; ++j) {
    int64_t pos = 0;
    if (s_idf[j] != 0.0 && s_wid[j] > 0 && strip0 > 0 && strip0 < p.n_docs)
      pos = warp_lower_bound(p.post_doc + s_lo[j], 0, s_n[j], (int32_t)strip0, lane);
    if (lane == 0) my_cur[j] = (int32_t)pos;
  }
  __syncwarp();

  const unsigned long long thr_key = MODE == kModeCollect ? p.thr[qi] : 0ull;
  const double td = orderable_f64(thr_key);
  for (int64_t s0l = strip0; s0l < strip0 + strip_len && s0l < p.n_docs; s0l += kSub) {
    const int32_t s0 = (int32_t)s0l;
    const int32_t s1 = (int32_t)min(s0l + kSub, p.n_docs);
    const int nd = s1 - s0;
    for (int j = 0; j < len; ++j) {
      const double w = s_idf[j];
      if (w == 0.0) continue;  // warp-uniform
      const int wid = s_wid[j];
      if (wid < 0) {
        // ---- head term: dense ratio row, every doc of the sub-range (0.0 where the doc has no posting)
        const double* __restrict__ dr = p.dense_ratio + (size_t)(-1 - wid) * p.n_docs + s0;
        double r[kSub / 32];
#pragma unroll
        for (int c = 0; c < kSub / 32; ++c) r[c] = (c * 32 + lane) < nd ? __ldg(dr + c * 32 + lane) : 0.0;
#pragma unroll
        for (int c = 0; c < kSub / 32; ++c) {
          const uint32_t ad = a_s + (uint32_t)(c * 32 + lane) * 8u;
          const double add = PLUS ? __dmul_rn(w, __dadd_rn(p.delta, r[c])) : __dmul_rn(w, r[c]);
          if ((c * 32 + lane) < nd) sts_f64(ad, __dadd_rn(lds_f64(ad), add));
        }
        __syncwarp();
        continue;
      }
      const int32_t n = s_n[j];
      const int32_t* __restrict__ pd = p.post_doc + s_lo[j];
      const double* __restrict__ pr = p.ratio + s_lo[j];
      int32_t cur = my_cur[j];
      // chunk loop, specialised on the number of 32-posting chunks in flight (warp-uniform).  The postings of the list are
      // sorted by doc, so the ones inside [s0, s1) are a prefix of what is fetched: their count advances the cursor.
      // Branch-free body: a posting beyond the sub-range reads the warp's (never written) dummy slot and stores nothing.
      auto walk = [&](auto width) {
        constexpr int W = decltype(width)::value;
        for (;;) {
          int32_t doc[W];
          double rat[W];
#pragma unroll
          for (int u = 0; u < W; ++u) {
            const int32_t i = cur + u * 32 + lane;
            const bool ok = i < n;
            doc[u] = ok ? __ldg(pd + (ok ? i : 0)) : 0x7fffffff;
            rat[u] = ok ? __ldg(pr + (ok ? i : 0)) : 0.0;
          }
          int inside = 0;
#pragma unroll
          for (int u = 0; u < W; ++u) {
            const bool in = doc[u] < s1;
            const uint32_t ad = in ? a_s + (uint32_t)(doc[u] - s0) * 8u : dummy_s;   // dummy: read-only, holds 0.0
            const double add = PLUS ? __dmul_rn(w, __dadd_rn(p.delta, rat[u])) : __dmul_rn(w, rat[u]);
            const double sum = __dadd_rn(lds_f64(ad), add);
            if (in) sts_f64(ad, sum);
            if (PLUS && in) atomicOr(&bits[(doc[u] - s0) >> 5], 1u << ((doc[u] - s0) & 31));
            inside += __popc(__ballot_sync(0xffffffffu, in));
          }
          cur += inside;
          if (inside < 32 * W) break;
        }
      };
      if (cur < n) {   // warp-uniform: the list still has postings at or beyond this sub-range
        if (wid == 1)
          walk(std::integral_constant<int, 1>());
        else
          walk(std::integral_constant<int, kRsPost>());
        if (lane == 0) my_cur[j] = cur;
      }
      __syncwarp();   // the next term's lanes may touch accumulators this term's other lanes just wrote
      if (PLUS) {
        // every doc of the sub-range WITHOUT a posting of this term gets idf * (delta + 0.0)
        const double wd = __dmul_rn(w, __dadd_rn(p.delta, 0.0));
#pragma unroll 4
        for (int c = 0; c < kSub / 32; ++c) {
          const uint32_t word = bits[c];
          const int i = c * 32 + lane;
          if (i < nd && !((word >> lane) & 1u)) a[i] = __dadd_rn(a[i], wd);
        }
        __syncwarp();
        if (lane < kSub / 32) bits[lane] = 0u;
        __syncwarp();
      }
    }
    // the sub-range is complete: consume it
    if (MODE == kModeDump) {
      double* out = p.dump + (size_t)qi * p.n_docs + s0;
      for (int i = lane; i < kSub; i += 32) {
        if (i < nd) out[i] = a[i];
        a[i] = 0.0;
      }
    } else if (MODE == kModeCollect) {
      // thr is the orderable image of a positive double (or of "every positive score"): for positive scores the key order
      // is the numeric order, so the filter compares doubles and only survivors are converted
      unsigned long long* ok = p.ckey + (size_t)qi * p.n_docs;
      uint32_t* oi = p.cidx + (size_t)qi * p.n_docs;
#pragma unroll 4
      for (int i = lane; i < kSub; i += 32) {
        const double sv = a[i];
        a[i] = 0.0;
        const bool pass = i < nd && sv > 0.0 && sv >= td && sv <= 1.7976931348623157e308;  // finite positive (NaN fails)
        const unsigned m = __ballot_sync(0xffffffffu, pass);
        if (m) {
          int at = 0;
          if (lane == 0) at = atomicAdd(&p.cnt[qi], __popc(m));
          at = __shfl_sync(0xffffffffu, at, 0);
          if (pass) {
            at += __popc(m & ((1u << lane) - 1u));
            ok[at] = f64_orderable(sv);
            oi[at] = (uint32_t)(s0 + i);
          }
        }
      }
    }
    __syncwarp();
  }
  if (MODE == kModeSample) {
    // the CTA's single range is scored (one sub-range per warp): its accumulators become sort keys in place
    __syncthreads();
    const int32_t r0 = (int32_t)(first * kRange);
    const int nd = (int)min((int64_t)kRange, p.n_docs - r0);
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(acc);
    if (tid == 0) npos = 0;
    __syncthreads();
    int local = 0;
    for (int i = tid; i < kRange; i += kRsThreads) {
      const double sc = acc[i];
      const unsigned long long key = (i < nd && sc > 0.0) ? f64_orderable(sc) : 0ull;
      keys[i] = key;
      local += key != 0ull;
    }
    local = __reduce_add_sync(0xffffffffu, local);
    if (lane == 0 && local) atomicAdd(&npos, local);
    __syncthreads();
    // S sample ranges each report their ceil(k / S)-th best positive score; at least k docs score >= the MINIMUM of
    // those, so it is a lower bound of the global k-th best (a range with too few positives degrades the bound to
    // "every positive score", never below).  thr[] was preset to all-ones by the host.
    unsigned long long t = kPosZero + 1ull;
    if (npos >= p.k) t = block_kth_largest(keys, kRange, p.k, hist, scal, 3);  // sign + exponent + 12 mantissa bits
    if (tid == 0) atomicMin(p.thr + qi, t);
  }
}

// ------------------------------------------------------------------------------------------------ top-k select
// Pair ordering: larger key first, ties -> smaller idx first.  key 0 == empty.
__device__ __forceinline__ bool pair_before(unsigned long long ka, uint32_t ia, unsigned long long kb, uint32_t ib) {
  return (ka > kb) || (ka == kb && ia < ib);
}

template <int NT>
__device__ __forceinline__ void block_bitonic_sort_pairs(unsigned long long* key, uint32_t* idx, int len, int tid) {
  for (int k = 2; k <= len; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < len; i += NT) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long a = key[i], b = key[ixj];
          const uint32_t ia = idx[i], ib = idx[ixj];
          const bool a_first = pair_before(a, ia, b, ib);
          const bool desc = (i & k) == 0;
          if ((desc ? !a_first : a_first) && !(a == b && ia == ib)) {
            key[i] = b; key[ixj] = a;
            idx[i] = ib; idx[ixj] = ia;
          }
        }
      }
      __syncthreads();
    }
  }
}

// ------------------------------------------------------------------------------------------------ top-k select v2
// sample threshold -> collect -> radix select.  (1) per query, the k-th best positive score among the first 8192 docs is a
// safe lower bound of the global k-th best; (2) one streaming pass collects every doc with score > 0 and >= bound
// (~ N * k / 8192 docs) into a per-query buffer sized for the worst case; (3) one CTA per query finds the k-th largest
// score by MSB-first radix select, breaks exact ties by ascending doc index with a second radix select, sorts the k
// winners.  Exact for any score distribution (an unrepresentative sample only enlarges step 2's output).
constexpr int kBmStage = 12288;  // (key, idx) pairs staged in shared memory by the final kernel (144 KB)

// K-th largest value among keys[0..n) (shared memory, every thread of the CTA participates); n >= K >= 1.
// passes < 8 stops after the leading 8 * passes bits and returns the LOWER EDGE of the bucket that holds the K-th largest
// key (<= the exact answer): all a safe threshold needs.
__device__ unsigned long long block_kth_largest(const unsigned long long* keys, int n, int K, int* hist, int* scal,
                                                int passes) {
  const int tid = threadIdx.x, nt = blockDim.x;
  unsigned long long prefix = 0ull, mask = 0ull;
  int need = K;
  for (int shift = 56; shift >= 0 && passes > 0; shift -= 8, --passes) {
    for (int i = tid; i < 256; i += nt) hist[i] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += nt) {
      const unsigned long long key = keys[i];
      if ((key & mask) == prefix) {  // warp-aggregated: equal digits elect one lane (concentrated digits serialise)
        const int dgt = (int)((key >> shift) & 0xffull);
        const unsigned grp = __match_any_sync(__activemask(), dgt);
        if ((int)(threadIdx.x & 31) == __ffs(grp) - 1) atomicAdd(&hist[dgt], __popc(grp));
      }
    }
    __syncthreads();
    if (tid < 32) warp_select_bin<true>(hist, need, tid, scal);
    __syncthreads();
    prefix |= (unsigned long long)scal[0] << shift;
    mask |= 0xffull << shift;
    need = scal[1];
    __syncthreads();
  }
  return prefix;
}

__global__ void __launch_bounds__(1024, 1) bm25_final_select_kernel(const unsigned long long* __restrict__ ckey,
                                                                    const uint32_t* __restrict__ cidx,
                                                                    const int32_t* __restrict__ cnt, int64_t n_docs,
                                                                    int k, int kpow2, int64_t id_base,
                                                                    int64_t* __restrict__ out_ids,
                                                                    double* __restrict__ out_scores,
                                                                    int32_t* __restrict__ out_counts) {
  extern __shared__ __align__(16) uint8_t fsm2[];
  unsigned long long* skey = reinterpret_cast<unsigned long long*>(fsm2);   // [kBmStage]
  uint32_t* sidx = reinterpret_cast<uint32_t*>(skey + kBmStage);            // [kBmStage]
  unsigned long long* wkey = reinterpret_cast<unsigned long long*>(sidx + kBmStage);  // [kpow2]
  uint32_t* widx = reinterpret_cast<uint32_t*>(wkey + kpow2);                           // [kpow2]
  __shared__ int hist[256];
  __shared__ int scal[4];
  const int qi = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
  const int n = cnt[qi];
  const unsigned long long* gk = ckey + (size_t)qi * n_docs;
  const uint32_t* gi = cidx + (size_t)qi * n_docs;
  const bool staged = n <= kBmStage;
  if (staged) {
    for (int i = tid; i < n; i += nt) {
      skey[i] = gk[i];
      sidx[i] = gi[i];
    }
  }
  const unsigned long long* K_ = staged ? skey : gk;
  const uint32_t* I_ = staged ? sidx : gi;
  __syncthreads();
  unsigned long long T = 0ull;        // k-th largest score key; winners: key > T, or key == T with idx <= Icut
  uint32_t Icut = 0xffffffffu;
  if (n > k) {
    // (a) k-th largest key
    unsigned long long prefix = 0ull, mask = 0ull;
    int need = k;
    for (int shift = 56; shift >= 0; shift -= 8) {
      for (int i = tid; i < 256; i += nt) hist[i] = 0;
      __syncthreads();
      for (int i = tid; i < n; i += nt) {
        const unsigned long long key = K_[i];
        if ((key & mask) == prefix) {
          const int dgt = (int)((key >> shift) & 0xffull);
          const unsigned grp = __match_any_sync(__activemask(), dgt);
          if ((int)(threadIdx.x & 31) == __ffs(grp) - 1) atomicAdd(&hist[dgt], __popc(grp));
        }
      }
      __syncthreads();
      if (tid < 32) warp_select_bin<true>(hist, need, tid, scal);
      __syncthreads();
      prefix |= (unsigned long long)scal[0] << shift;
      mask |= 0xffull << shift;
      need = scal[1];
      __syncthreads();
    }
    T = prefix;
    const int m = need;  // how many docs with key == T belong to the top k (1 <= m <= #equal)
    // (b) m-th smallest doc index among key == T
    uint32_t ipre = 0u, imask = 0u;
    int ineed = m;
    for (int shift = 24; shift >= 0; shift -= 8) {
      for (int i = tid; i < 256; i += nt) hist[i] = 0;
      __syncthreads();
      for (int i = tid; i < n; i += nt) {
        if (K_[i] == T) {
          const uint32_t ix = I_[i];
          if ((ix & imask) == ipre) atomicAdd(&hist[(int)((ix >> shift) & 0xffu)], 1);
        }
      }
      __syncthreads();
      if (tid < 32) warp_select_bin<false>(hist, ineed, tid, scal);
      __syncthreads();
      ipre |= (uint32_t)scal[0] << shift;
      imask |= 0xffu << shift;
      ineed = scal[1];
      __syncthreads();
    }
    Icut = ipre;
  }
  // gather the winners, then order them (score desc, doc asc)
  if (tid == 0) scal[2] = 0;
  for (int i = tid; i < kpow2; i += nt) {
    wkey[i] = 0ull;
    widx[i] = 0xffffffffu;
  }
  __syncthreads();
  for (int i = tid; i < n; i += nt) {
    const unsigned long long key = K_[i];
    const uint32_t ix = I_[i];
    if (key > T || (key == T && ix <= Icut)) {
      const int at = atomicAdd(&scal[2], 1);
      if (at < kpow2) {
        wkey[at] = key;
        widx[at] = ix;
      }
    }
  }
  __syncthreads();
  block_bitonic_sort_pairs<1024>(wkey, widx, kpow2, tid);
  const int nw = min(min(scal[2], k), kpow2);
  for (int i = tid; i < k; i += nt) {
    const bool valid = i < nw;
    out_ids[(size_t)qi * k + i] = valid ? id_base + (int64_t)widx[i] : -1;
    out_scores[(size_t)qi * k + i] = valid ? orderable_f64(wkey[i]) : 0.0;
  }
  if (tid == 0) out_counts[qi] = nw;
}

int pow2_at_least(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

size_t range_smem_bytes(int max_len) {
  return (size_t)kRange * 8 + kRsWarps * 8 + (size_t)std::max(max_len, 1) * (8 + 8 + 4 + 4 + 4 * kRsWarps) + (kRange / 32) * 4 + 16;
}

template <int MODE, bool PLUS>
int launch_range_kernel(sb_ctx* ctx, const RangeParams& rp, int nq, int n_chunks, cudaStream_t st) {
  const size_t smem = range_smem_bytes(rp.max_len);
  SB_REQUIRE(smem <= ctx->smem_optin, SB_ERR_UNSUPPORTED, "bm25: a query of %d terms does not fit the per-CTA term state",
             rp.max_len);
  SB_CUDA(cudaFuncSetAttribute(bm25_range_kernel<MODE, PLUS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  bm25_range_kernel<MODE, PLUS><<<dim3((unsigned)nq, (unsigned)n_chunks), kRsThreads, smem, st>>>(rp);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

template <int MODE>
int launch_range(sb_ctx* ctx, const RangeParams& rp, int nq, int n_chunks, cudaStream_t st) {
  return ctx->bm25.variant == SB_BM25_PLUS ? launch_range_kernel<MODE, true>(ctx, rp, nq, n_chunks, st)
                                           : launch_range_kernel<MODE, false>(ctx, rp, nq, n_chunks, st);
}

RangeParams range_params(sb_ctx* ctx, const int32_t* q_terms_dev, const int32_t* q_off_dev, int max_len) {
  const Bm25Index& ix = ctx->bm25;
  RangeParams rp;
  memset(&rp, 0, sizeof(rp));
  rp.q_terms = q_terms_dev;
  rp.q_off = q_off_dev;
  rp.max_len = std::max(max_len, 1);
  rp.ranges_per_cta = 1;
  rp.indptr = ix.indptr;
  rp.post_doc = ix.post_doc;
  rp.ratio = ix.post_ratio;
  rp.idf = ix.idf;
  rp.dense_of_term = ix.n_dense > 0 ? ix.dense_of_term : nullptr;
  rp.dense_ratio = ix.dense_ratio;
  rp.n_terms = ix.n_terms;
  rp.n_docs = ix.n_docs;
  rp.delta = ix.delta;
  return rp;
}

// consecutive ranges per CTA: long runs amortise the per-term posting-list search, short runs fill the machine
int ranges_per_cta(sb_ctx* ctx, int nq, int64_t n_ranges) {
  const int64_t resident = (int64_t)ctx->num_sms * 2;  // 2 CTAs of bm25_range_kernel per SM (64 registers per thread)
  int64_t r = ((int64_t)nq * n_ranges) / (resident * 2);   // about two waves of CTAs: long strips, balanced tail
  if (r < 1) r = 1;
  if (r > 32) r = 32;
  return (int)r;
}

int bm25_topk_enqueue(sb_ctx* ctx, const int32_t* q_terms_dev, const int32_t* q_off_dev, int B, int max_len, int k,
                      int64_t* out_ids, double* out_scores, int32_t* out_counts, cudaStream_t st) {
  Bm25Index& ix = ctx->bm25;
  const int kpow2 = std::max(32, pow2_at_least(k));
  SB_REQUIRE(kpow2 <= 1024, SB_ERR_UNSUPPORTED, "bm25: top_k %d too large (max 1024)", k);
  // sub-batch: the worst-case candidate lists ((key, idx) per doc per query) of a sub-batch stay under 1.5 GB
  int64_t sbq = (int64_t)((1536ull << 20) / ((size_t)ix.n_docs * 12 + 1));
  sbq = std::max<int64_t>(1, std::min<int64_t>(sbq, B));
  int rc;
  if ((rc = ctx->misc2_dev.reserve((size_t)sbq * ix.n_docs * 8 + (size_t)sbq * 16 + 64))) return rc;
  if ((rc = ctx->misc3_dev.reserve((size_t)sbq * ix.n_docs * 4 + 64))) return rc;
  unsigned long long* ckey = ctx->misc2_dev.as<unsigned long long>();
  unsigned long long* thr = ckey + (size_t)sbq * ix.n_docs;
  int32_t* cnt = reinterpret_cast<int32_t*>(thr + sbq);
  uint32_t* cidx = ctx->misc3_dev.as<uint32_t>();
  const size_t fin_smem = (size_t)kBmStage * 12 + (size_t)kpow2 * 12 + 64;
  SB_CUDA(cudaFuncSetAttribute(bm25_final_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fin_smem));
  const int64_t n_ranges = (ix.n_docs + kRange - 1) / kRange;
  for (int b0 = 0; b0 < B; b0 += (int)sbq) {
    const int nq = (int)std::min<int64_t>(sbq, B - b0);
    RangeParams rp = range_params(ctx, q_terms_dev, q_off_dev + b0, max_len);
    rp.k = k;
    rp.thr = thr;
    rp.cnt = cnt;
    rp.ckey = ckey;
    rp.cidx = cidx;
    {
      ProfScope ps(ctx, SB_PROF_BM25_SCORE, st, 2);
      // (1) safe per-query lower bound of the k-th best score from S sample ranges (exact k-th best when S == 1)
      // (4 sample ranges: a sample CTA pays the full per-warp set-up -- one posting-list search per term -- for a single
      // sub-range, so 8 of them cost 21 % of the collect pass for 6.5 % of its docs; a lower bound from 4 is nearly as tight)
      const int S = (int)std::min<int64_t>(4, n_ranges);
      rp.k = (k + S - 1) / S;
      SB_CUDA(cudaMemsetAsync(thr, 0xff, (size_t)nq * 8, st));
      SB_CUDA(cudaMemsetAsync(cnt, 0, (size_t)nq * 4, st));
      if ((rc = launch_range<kModeSample>(ctx, rp, nq, S, st))) return rc;
      // (2) score every range in shared memory, keep only docs that can still reach the top k
      rp.ranges_per_cta = ranges_per_cta(ctx, nq, n_ranges);
      const int n_chunks = (int)((n_ranges + rp.ranges_per_cta - 1) / rp.ranges_per_cta);
      if ((rc = launch_range<kModeCollect>(ctx, rp, nq, n_chunks, st))) return rc;
    }
    ProfScope ps(ctx, SB_PROF_BM25_SELECT, st, 1);
    // (3) exact k-th largest by radix select over the (few) candidates, ties by ascending doc index, sort the winners
    bm25_final_select_kernel<<<nq, 1024, fin_smem, st>>>(ckey, cidx, cnt, ix.n_docs, k, kpow2, ix.id_base,
                                                         out_ids + (size_t)b0 * k, out_scores + (size_t)b0 * k,
                                                         out_counts + b0);
    SB_CUDA(cudaGetLastError());
  }
  return SB_OK;
}

__global__ void bm25_fill_empty_kernel(int64_t* ids, double* sc, int32_t* cnt, int B, int k) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B * k) {
    ids[i] = -1;
    sc[i] = 0.0;
  }
  if (i < B) cnt[i] = 0;
}

}  // namespace

// Installs a term-major CSR that already lives on the device as the context's BM25 index (sb_bm25_load uploads host
// arrays first; the GPU builder of bm25_build.cu hands its arrays over directly).  Takes ownership of indptr_dev and
// post_doc_dev; tf_dev / doc_len_dev are only read (dnorm and the query-independent ratio are derived from them).
static void bm25_index_free(Bm25Index& ix) {
  if (ix.indptr) cudaFree(ix.indptr);
  if (ix.post_doc) cudaFree(ix.post_doc);
  if (ix.post_ratio) cudaFree(ix.post_ratio);
  if (ix.dnorm) cudaFree(ix.dnorm);
  if (ix.idf) cudaFree(ix.idf);
  if (ix.dense_of_term) cudaFree(ix.dense_of_term);
  if (ix.dense_ratio) cudaFree(ix.dense_ratio);
  ix = Bm25Index();
}

// The new index is assembled in a local object and swapped in only when every allocation and kernel has succeeded: a failed
// load leaves the context with its previous index intact (and frees everything it took ownership of).
static int bm25_install_build(Bm25Index& nx, const uint16_t* tf_dev, const int32_t* doc_len_dev, const double* idf_host,
                              cudaStream_t st) {
  SB_CUDA(cudaMalloc(&nx.idf, (size_t)std::max<int64_t>(nx.n_terms, 1) * 8));
  if (nx.n_terms) SB_CUDA(cudaMemcpyAsync(nx.idf, idf_host, (size_t)nx.n_terms * 8, cudaMemcpyHostToDevice, st));
  SB_CUDA(cudaMalloc(&nx.dnorm, (size_t)std::max<int64_t>(nx.n_docs, 1) * 8));
  // query-independent fp64 ratio tf*(k1+1)/(tf+dnorm[doc]) (8 B per posting) replaces the 2 B tf + 8 B dnorm gather
  SB_CUDA(cudaMalloc(&nx.post_ratio, (size_t)std::max<int64_t>(nx.nnz, 1) * 8));
  if (nx.n_docs) {
    const double omb = 1.0 - nx.b;  // Python evaluates `1 - self.b` first (left-to-right)
    bm25_dnorm_kernel<<<(unsigned)((nx.n_docs + 255) / 256), 256, 0, st>>>(doc_len_dev, nx.n_docs, nx.k1, nx.b, omb,
                                                                          nx.avgdl, nx.dnorm);
    SB_CUDA(cudaGetLastError());
  }
  if (nx.nnz) {
    const double k1p1 = nx.k1 + 1.0;
    bm25_ratio_kernel<<<(unsigned)((nx.nnz + 255) / 256), 256, 0, st>>>(nx.post_doc, tf_dev, nx.nnz, nx.dnorm, k1p1,
                                                                       nx.post_ratio);
    SB_CUDA(cudaGetLastError());
  }
  SB_CUDA(cudaStreamSynchronize(st));
  // dense ratio rows of the head terms (df >= n_docs / 4): at most 64 rows and 2 GB
  if (nx.n_terms > 0 && nx.n_docs >= 4096) {
    std::vector<int64_t> indptr_h((size_t)nx.n_terms + 1);
    SB_CUDA(cudaMemcpy(indptr_h.data(), nx.indptr, indptr_h.size() * 8, cudaMemcpyDeviceToHost));
    std::vector<std::pair<int64_t, int32_t>> heavy;   // (df, term)
    for (int64_t t = 0; t < nx.n_terms; ++t) {
      const int64_t df = indptr_h[(size_t)t + 1] - indptr_h[(size_t)t];
      if (df * 4 >= nx.n_docs) heavy.push_back({df, (int32_t)t});
    }
    std::sort(heavy.begin(), heavy.end(), [](const auto& a, const auto& b) { return a.first > b.first; });
    const size_t row_bytes = (size_t)nx.n_docs * 8;
    const size_t max_rows = std::min<size_t>(64, (size_t)(2048ull << 20) / row_bytes);
    if (heavy.size() > max_rows) heavy.resize(max_rows);
    if (!heavy.empty()) {
      std::vector<int32_t> of_term((size_t)nx.n_terms, -1), slot_term(heavy.size());
      for (size_t sidx = 0; sidx < heavy.size(); ++sidx) {
        of_term[(size_t)heavy[sidx].second] = (int32_t)sidx;
        slot_term[sidx] = heavy[sidx].second;
      }
      int32_t* slot_term_dev = nullptr;
      SB_CUDA(cudaMalloc(&nx.dense_of_term, of_term.size() * 4));
      SB_CUDA(cudaMalloc(&nx.dense_ratio, heavy.size() * row_bytes));
      SB_CUDA(cudaMalloc(&slot_term_dev, slot_term.size() * 4));
      SB_CUDA(cudaMemcpyAsync(nx.dense_of_term, of_term.data(), of_term.size() * 4, cudaMemcpyHostToDevice, st));
      SB_CUDA(cudaMemcpyAsync(slot_term_dev, slot_term.data(), slot_term.size() * 4, cudaMemcpyHostToDevice, st));
      SB_CUDA(cudaMemsetAsync(nx.dense_ratio, 0, heavy.size() * row_bytes, st));
      bm25_dense_fill_kernel<<<dim3(256, (unsigned)heavy.size()), 256, 0, st>>>(nx.indptr, nx.post_doc, nx.post_ratio,
                                                                                slot_term_dev, nx.n_docs, nx.dense_ratio);
      cudaError_t fe = cudaGetLastError();
      cudaStreamSynchronize(st);
      cudaFree(slot_term_dev);
      SB_CUDA(fe);
      nx.n_dense = (int32_t)heavy.size();
    }
  }
  return SB_OK;
}

int bm25_install_device_csr(sb_ctx* ctx, int64_t* indptr_dev, int32_t* post_doc_dev, const uint16_t* tf_dev,
                            const int32_t* doc_len_dev, int64_t n_terms, int64_t nnz, int64_t n_docs, double avgdl,
                            const double* idf_host, int32_t variant, double k1, double b, double delta, int64_t id_base,
                            cudaStream_t st) {
  Bm25Index nx;
  nx.n_docs = n_docs;
  nx.n_terms = n_terms;
  nx.nnz = nnz;
  nx.id_base = id_base;
  nx.variant = variant;
  nx.k1 = k1;
  nx.b = b;
  nx.delta = delta;
  nx.avgdl = avgdl;
  nx.indptr = indptr_dev;      // ownership taken here, whatever happens next
  nx.post_doc = post_doc_dev;
  const int rc = bm25_install_build(nx, tf_dev, doc_len_dev, idf_host, st);
  if (rc != SB_OK) {
    cudaStreamSynchronize(st);
    bm25_index_free(nx);
    return rc;
  }
  cudaStreamSynchronize(st);   // nothing queued may still read the index that is about to be released
  bm25_index_free(ctx->bm25);
  ctx->bm25 = nx;
  return SB_OK;
}

extern "C" {

int sb_bm25_load(sb_ctx* ctx, const int64_t* indptr, const int32_t* post_doc, const uint16_t* post_tf,
                 int64_t n_terms, int64_t nnz, const int32_t* doc_len, int64_t n_docs, double avgdl,
                 const double* idf, int32_t variant, double k1, double b, double delta, int64_t id_base) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_bm25_load: ctx is NULL");
  SB_REQUIRE(n_terms >= 0 && nnz >= 0 && n_docs >= 0, SB_ERR_ARG, "sb_bm25_load: negative size");
  SB_REQUIRE(n_docs < (1ll << 31), SB_ERR_ARG, "sb_bm25_load: a shard holds at most 2^31-1 docs");
  SB_REQUIRE(variant == SB_BM25_OKAPI || variant == SB_BM25_PLUS, SB_ERR_ARG, "sb_bm25_load: bad variant %d", variant);
  SB_REQUIRE(indptr && (nnz == 0 || (post_doc && post_tf)) && (n_docs == 0 || doc_len) && (n_terms == 0 || idf),
             SB_ERR_ARG, "sb_bm25_load: NULL buffer");
  SB_REQUIRE(indptr[0] == 0 && indptr[n_terms] == nnz, SB_ERR_ARG, "sb_bm25_load: indptr does not span nnz");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  cudaStream_t st = ctx->stream;
  SB_CUDA(cudaStreamSynchronize(st));
  int64_t* indptr_dev = nullptr;
  int32_t* post_doc_dev = nullptr;
  auto stage = [&]() -> int {
    SB_CUDA(cudaMalloc(&indptr_dev, (size_t)(n_terms + 1) * 8));
    SB_CUDA(cudaMemcpyAsync(indptr_dev, indptr, (size_t)(n_terms + 1) * 8, cudaMemcpyHostToDevice, st));
    SB_CUDA(cudaMalloc(&post_doc_dev, (size_t)std::max<int64_t>(nnz, 1) * 4));
    int rc;
    if ((rc = ctx->misc_dev.reserve((size_t)std::max<int64_t>(n_docs, 1) * 4))) return rc;
    if ((rc = ctx->misc2_dev.reserve((size_t)std::max<int64_t>(nnz, 1) * 2))) return rc;
    if (n_docs) SB_CUDA(cudaMemcpyAsync(ctx->misc_dev.p, doc_len, (size_t)n_docs * 4, cudaMemcpyHostToDevice, st));
    if (nnz) {
      SB_CUDA(cudaMemcpyAsync(post_doc_dev, post_doc, (size_t)nnz * 4, cudaMemcpyHostToDevice, st));
      SB_CUDA(cudaMemcpyAsync(ctx->misc2_dev.p, post_tf, (size_t)nnz * 2, cudaMemcpyHostToDevice, st));
    }
    return SB_OK;
  };
  if (int rc = stage()) {  // nothing has taken ownership yet
    cudaStreamSynchronize(st);
    if (indptr_dev) cudaFree(indptr_dev);
    if (post_doc_dev) cudaFree(post_doc_dev);
    return rc;
  }
  return bm25_install_device_csr(ctx, indptr_dev, post_doc_dev, ctx->misc2_dev.as<uint16_t>(), ctx->misc_dev.as<int32_t>(),
                                 n_terms, nnz, n_docs, avgdl, idf, variant, k1, b, delta, id_base, st);
}

int64_t sb_bm25_count(sb_ctx* ctx) { return ctx ? ctx->bm25.n_docs : -1; }

int sb_bm25_topk_dev(sb_ctx* ctx, const int32_t* q_terms_dev, const int32_t* q_off_dev, int32_t B, int32_t n_q_terms,
                     int32_t max_q_len, int32_t k, int64_t* out_ids_dev, double* out_scores_dev,
                     int32_t* out_counts_dev, void* stream) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_bm25_topk_dev: ctx is NULL");
  SB_REQUIRE(B >= 0 && k > 0 && max_q_len >= 0 && n_q_terms >= 0, SB_ERR_ARG, "sb_bm25_topk_dev: bad sizes");
  if (B == 0) return SB_OK;
  SB_REQUIRE(q_off_dev && out_ids_dev && out_scores_dev && out_counts_dev, SB_ERR_ARG, "sb_bm25_topk_dev: NULL buffer");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  cudaStream_t st = pick_stream(ctx, stream);
  if (ctx->bm25.n_docs == 0 || ctx->bm25.indptr == nullptr) {
    bm25_fill_empty_kernel<<<(B * k + 255) / 256, 256, 0, st>>>(out_ids_dev, out_scores_dev, out_counts_dev, B, k);
    SB_CUDA(cudaGetLastError());
    return SB_OK;
  }
  return bm25_topk_enqueue(ctx, q_terms_dev, q_off_dev, B, max_q_len, k, out_ids_dev, out_scores_dev, out_counts_dev,
                           st);
}

int sb_bm25_topk(sb_ctx* ctx, const int32_t* q_terms, const int32_t* q_off, int32_t B, int32_t k, int64_t* out_ids,
                 double* out_scores, int32_t* out_counts) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_bm25_topk: ctx is NULL");
  SB_REQUIRE(B >= 0 && k > 0, SB_ERR_ARG, "sb_bm25_topk: bad B=%d k=%d", B, k);
  if (B == 0) return SB_OK;
  SB_REQUIRE(q_off && out_ids && out_scores && out_counts, SB_ERR_ARG, "sb_bm25_topk: NULL buffer");
  const int n_terms_q = q_off[B];
  SB_REQUIRE(n_terms_q >= 0 && (n_terms_q == 0 || q_terms), SB_ERR_ARG, "sb_bm25_topk: bad query term buffers");
  int max_len = 0;
  for (int b = 0; b < B; ++b) {
    SB_REQUIRE(q_off[b + 1] >= q_off[b], SB_ERR_ARG, "sb_bm25_topk: q_off must be non-decreasing");
    max_len = std::max(max_len, q_off[b + 1] - q_off[b]);
  }
  std::unique_lock<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  cudaStream_t st = ctx->stream;
  if (ctx->bm25.n_docs == 0 || ctx->bm25.indptr == nullptr) {
    for (int i = 0; i < B * k; ++i) { out_ids[i] = -1; out_scores[i] = 0.0; }
    for (int i = 0; i < B; ++i) out_counts[i] = 0;
    return SB_OK;
  }
  int rc;
  const size_t tb = (size_t)std::max(n_terms_q, 1) * 4, ob = (size_t)(B + 1) * 4;
  if ((rc = ctx->pin_in.reserve(tb + ob))) return rc;
  if ((rc = ctx->q_dev.reserve(tb + ob))) return rc;
  uint8_t* pi = ctx->pin_in.as<uint8_t>();
  if (n_terms_q) memcpy(pi, q_terms, (size_t)n_terms_q * 4);
  memcpy(pi + tb, q_off, ob);
  SB_CUDA(cudaMemcpyAsync(ctx->q_dev.p, pi, tb + ob, cudaMemcpyHostToDevice, st));
  const int32_t* qt_dev = ctx->q_dev.as<int32_t>();
  const int32_t* qo_dev = reinterpret_cast<const int32_t*>(ctx->q_dev.as<uint8_t>() + tb);
  const size_t nid = (size_t)B * k;
  if ((rc = ctx->out_ids_dev.reserve(nid * 8))) return rc;
  if ((rc = ctx->out_sc_dev.reserve(nid * 8))) return rc;
  if ((rc = ctx->out_cnt_dev.reserve((size_t)B * 4))) return rc;
  if ((rc = bm25_topk_enqueue(ctx, qt_dev, qo_dev, B, max_len, k, ctx->out_ids_dev.as<int64_t>(),
                              ctx->out_sc_dev.as<double>(), ctx->out_cnt_dev.as<int32_t>(), st)))
    return rc;
  if ((rc = ctx->pin_out.reserve(nid * 16 + (size_t)B * 4))) return rc;
  uint8_t* po = ctx->pin_out.as<uint8_t>();
  SB_CUDA(cudaMemcpyAsync(po, ctx->out_ids_dev.p, nid * 8, cudaMemcpyDeviceToHost, st));
  SB_CUDA(cudaMemcpyAsync(po + nid * 8, ctx->out_sc_dev.p, nid * 8, cudaMemcpyDeviceToHost, st));
  SB_CUDA(cudaMemcpyAsync(po + nid * 16, ctx->out_cnt_dev.p, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
  SB_CUDA(cudaStreamSynchronize(st));
  memcpy(out_ids, po, nid * 8);
  memcpy(out_scores, po + nid * 8, nid * 8);
  memcpy(out_counts, po + nid * 16, (size_t)B * 4);
  return SB_OK;
}

int sb_bm25_scores(sb_ctx* ctx, const int32_t* q_terms, int32_t n_q, double* out_scores) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_bm25_scores: ctx is NULL");
  SB_REQUIRE(n_q >= 0 && (n_q == 0 || q_terms) && out_scores, SB_ERR_ARG, "sb_bm25_scores: bad arguments");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  Bm25Index& ix = ctx->bm25;
  SB_REQUIRE(ix.indptr != nullptr, SB_ERR_STATE, "sb_bm25_scores: no BM25 index loaded");
  if (ix.n_docs == 0) return SB_OK;
  cudaStream_t st = ctx->stream;
  int rc;
  const size_t tb = (size_t)std::max(n_q, 1) * 4;
  if ((rc = ctx->q_dev.reserve(tb + 8))) return rc;
  int32_t off[2] = {0, n_q};
  if (n_q) SB_CUDA(cudaMemcpyAsync(ctx->q_dev.p, q_terms, (size_t)n_q * 4, cudaMemcpyHostToDevice, st));
  SB_CUDA(cudaMemcpyAsync(ctx->q_dev.as<uint8_t>() + tb, off, 8, cudaMemcpyHostToDevice, st));
  if ((rc = ctx->acc_dev.reserve((size_t)ix.n_docs * sizeof(double)))) return rc;
  RangeParams rp = range_params(ctx, ctx->q_dev.as<int32_t>(),
                                reinterpret_cast<const int32_t*>(ctx->q_dev.as<uint8_t>() + tb), n_q);
  rp.dump = ctx->acc_dev.as<double>();
  const int64_t n_ranges = (ix.n_docs + kRange - 1) / kRange;
  rp.ranges_per_cta = ranges_per_cta(ctx, 1, n_ranges);
  ctx->launches += 1;
  if ((rc = launch_range<kModeDump>(ctx, rp, 1, (int)((n_ranges + rp.ranges_per_cta - 1) / rp.ranges_per_cta), st)))
    return rc;
  SB_CUDA(cudaMemcpyAsync(out_scores, ctx->acc_dev.p, (size_t)ix.n_docs * 8, cudaMemcpyDeviceToHost, st));
  SB_CUDA(cudaStreamSynchronize(st));
  return SB_OK;
}

}  // extern "C"
