// dense.cu -- K1: brute-force cosine top-k over an HBM-resident fp16 corpus.
//
// Replaces the Qdrant `client.search(...)` behind DenseRetriever.retrieve (reference src/core/retrievers/dense.py:41-64).
//
// Pipeline per pass of QB (1/2/4) queries:
//   dense_scan_kernel   persistent, one CTA per SM.  A producer warp streams row tiles HBM -> smem with 1-D bulk
//                       async copies (cp.async.bulk, the TMA engine; SASS UBLKCP) through an mbarrier ring; 8 consumer
//                       warps compute fp32 dot products (queries live in registers), apply the stored inverse row norm
//                       and push candidates that beat the CTA's running K'-th best into a smem candidate buffer that
//                       is compacted by an in-smem bitonic sort.  Output: one sorted top-K' list per CTA per query
//                       (K' = k + slack, power of two).
//   dense_merge_kernel  one CTA per query: the k-th best approximate key over the per-CTA lists, then EVERY row inside
//                       the error window below it (dense_common.cuh) is re-scored in fp64 against the STORED fp16 rows,
//                       final sort by (score desc, id asc), write k.  Queries whose window cannot be served from the
//                       lists raise a flag and are answered by dense_exact_fallback_kernel (brute force, fp64).
//
// Algorithmic HBM bytes per pass = n_pad * d_pad * 2 (+ n_pad * 4 for the inverse norms); see DESIGN.md.
#include <math.h>
#include <string.h>
#include <algorithm>

#include "dense_common.cuh"
#include "dense_mma.cuh"

namespace {

constexpr int kConsumerWarps = 8;
constexpr int kConsumerThreads = kConsumerWarps * 32;
constexpr int kScanThreads = kConsumerThreads + 64;  // + 1 TMA producer warp + 1 compaction warp
constexpr int kMergeThreads = 512;
constexpr int kRowPad = 128;  // n_pad granularity (tile rows of the tcgen05 scan; multiple of the CUDA-core tiles)

// ------------------------------------------------------------------------------------------------ load kernels
// One warp per row.  f32 input: x16 = fp16(x / ||x||) (division in fp64, single rounding); f16 input: verbatim.
// inv_norm = 1/||x16|| of the stored values (fp64 accumulate), 0 for all-zero rows.
template <typename TIn>
__global__ void dense_store_rows_kernel(const TIn* __restrict__ in, int64_t n_rows, int32_t d, int32_t d_pad,
                                        __half* __restrict__ rows, float* __restrict__ inv_norm, int64_t row0,
                                        bool normalise) {
  int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (r >= n_rows) return;
  const TIn* src = in + r * (int64_t)d;
  __half* dst = rows + (row0 + r) * (int64_t)d_pad;
  double scale = 1.0;
  if (normalise) {
    double ss = 0.0;
    for (int i = lane; i < d; i += 32) {
      double v = (double)(float)src[i];
      ss += v * v;
    }
    for (int o = 16; o; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    scale = ss > 0.0 ? sqrt(ss) : 1.0;
  }
  double ss16 = 0.0;
  for (int i = lane; i < d_pad; i += 32) {
    __half h = __float2half(0.f);
    if (i < d) {
      double v = (double)(float)src[i];
      h = normalise ? __double2half(v / scale) : __float2half((float)v);
    }
    dst[i] = h;
    double hv = (double)__half2float(h);
    ss16 += hv * hv;
  }
  for (int o = 16; o; o >>= 1) ss16 += __shfl_xor_sync(0xffffffffu, ss16, o);
  if (lane == 0) inv_norm[row0 + r] = ss16 > 0.0 ? (float)(1.0 / sqrt(ss16)) : 0.f;
}

// ------------------------------------------------------------------------------------------------ scan kernel
struct ScanParams {
  const __half* rows;
  const float* inv_norm;
  const float* q;            // [QB][d_pad] fp32 (zero padded) for THIS pass
  unsigned long long* cand;  // [QB][grid][kprime] composite keys, sorted descending per list
  int64_t n;                 // valid rows
  int32_t d_pad;
  int32_t ch;                // 16-byte chunks per row = d_pad / 8
  int32_t num_tiles;
  int32_t kprime;
  int32_t bcap;              // capacity of each of the two append batches per query (kprime + bcap = sort size)
  int32_t stages;
  uint32_t tile_bytes;
};

// Sum V per-lane partials across the warp: afterwards the lanes with (lane % (32/V)) == 0 hold value index lane/(32/V).
template <int V>
__device__ __forceinline__ float warp_reduce_multi(float (&v)[V], int lane) {
  int off = 16;
#pragma unroll
  for (int half = V / 2; half >= 1; half >>= 1) {
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int t = 0; t < half; ++t) {
      float send = upper ? v[t] : v[t + half];
      float keep = upper ? v[t + half] : v[t];
      v[t] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
    off >>= 1;
  }
  float r = v[0];
  for (; off >= 1; off >>= 1) r += __shfl_xor_sync(0xffffffffu, r, off);
  return r;
}

// ---- asynchronous compaction (runs on its own warp, off the FMA warps' critical path) -------------------------------
// Descending bitonic sort of T = 32 * NPER 64-bit keys held in registers across one warp; element e = lane * NPER + r.
template <int NPER>
__device__ __forceinline__ void warp_sort_desc(unsigned long long (&v)[NPER], int lane) {
  constexpr int T = NPER * 32;
#pragma unroll
  for (int k = 2; k <= T; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (j < NPER) {
#pragma unroll
        for (int r = 0; r < NPER; ++r) {
          const int pr = r ^ j;
          if (pr > r) {
            const bool desc = (k < NPER) ? ((r & k) == 0) : ((lane & (k / NPER)) == 0);
            const unsigned long long x = v[r], y = v[pr];
            const bool sw = desc ? (x < y) : (x > y);
            v[r] = sw ? y : x;
            v[pr] = sw ? x : y;
          }
        }
      } else {
        const int lj = j / NPER;
        const bool lower = (lane & lj) == 0;
        const bool desc = (lane & (k / NPER)) == 0;
        const bool keep_max = lower == desc;
#pragma unroll
        for (int r = 0; r < NPER; ++r) {
          const unsigned long long o = __shfl_xor_sync(0xffffffffu, v[r], lj);
          const unsigned long long x = v[r];
          v[r] = keep_max ? (x > o ? x : o) : (x < o ? x : o);
        }
      }
    }
  }
}

// best[0..nbest) U batch[0..nbatch)  ->  best[0..min(K', nbest+nbatch))  (sorted descending); returns the new count.
template <int NPER>
__device__ __noinline__ int compact_into_best(unsigned long long* best, int nbest, const unsigned long long* batch,
                                              int nbatch, int kprime, int lane) {
  unsigned long long v[NPER];
#pragma unroll
  for (int r = 0; r < NPER; ++r) {
    const int e = lane * NPER + r;
    unsigned long long x = 0ull;
    if (e < nbest) x = best[e];
    else if (e - nbest < nbatch) x = batch[e - nbest];
    v[r] = x;
  }
  __syncwarp();
  warp_sort_desc<NPER>(v, lane);
#pragma unroll
  for (int r = 0; r < NPER; ++r) {
    const int e = lane * NPER + r;
    if (e < kprime) best[e] = v[r];
  }
  __syncwarp();
  const int total = nbest + nbatch;
  return total < kprime ? total : kprime;
}

// Generic (k > 100) path: same result through a shared-memory scratch of T keys, loop-based warp bitonic sort.
__device__ __noinline__ int compact_into_best_smem(unsigned long long* best, int nbest, const unsigned long long* batch,
                                                   int nbatch, int kprime, int T, unsigned long long* scratch,
                                                   int lane) {
  for (int e = lane; e < T; e += 32) {
    unsigned long long x = 0ull;
    if (e < nbest) x = best[e];
    else if (e - nbest < nbatch) x = batch[e - nbest];
    scratch[e] = x;
  }
  __syncwarp();
  for (int k = 2; k <= T; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = lane; i < T; i += 32) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long x = scratch[i], y = scratch[ixj];
          const bool desc = (i & k) == 0;
          if (desc ? (x < y) : (x > y)) {
            scratch[i] = y;
            scratch[ixj] = x;
          }
        }
      }
      __syncwarp();
    }
  }
  for (int e = lane; e < kprime; e += 32) best[e] = scratch[e];
  __syncwarp();
  const int total = nbest + nbatch;
  return total < kprime ? total : kprime;
}

__device__ __forceinline__ int compact_dispatch(int T, unsigned long long* best, int nbest,
                                                const unsigned long long* batch, int nbatch, int kprime,
                                                unsigned long long* scratch, int lane) {
  if (T == 512) return compact_into_best<16>(best, nbest, batch, nbatch, kprime, lane);
  return compact_into_best_smem(best, nbest, batch, nbatch, kprime, T, scratch, lane);
}

// two fp32 FMAs per instruction (SASS FFMA2): the 3-register FFMA issues at half rate on sm_100, FFMA2 restores
// the full 128 FMA/clk/SM; operands are (lo, hi) float pairs packed in 64-bit registers.
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ unsigned long long pack_f2(float lo, float hi) {
  return ((unsigned long long)__float_as_uint(hi) << 32) | (unsigned long long)__float_as_uint(lo);
}
__device__ __forceinline__ unsigned long long h2_to_f2(uint32_t h2) {
  const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&h2));
  return pack_f2(f.x, f.y);
}

template <int NCHUNK, int QB, int RW, bool EXACT>
__global__ void __launch_bounds__(kScanThreads, 1) dense_scan_kernel(const ScanParams p) {
  constexpr int R = kConsumerWarps * RW;  // rows per tile
  constexpr int V = RW * QB;              // partial sums per lane
  constexpr int LPV = 32 / V;             // lanes per value after the reduction
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* tiles = smem;
  // per query: best[K'] (sorted, owned by the compaction warp) + two append batches of bcap keys (ping / pong)
  const int qstride = p.kprime + 2 * p.bcap;
  unsigned long long* cbuf = reinterpret_cast<unsigned long long*>(smem + (size_t)p.stages * p.tile_bytes);
  const int scratch_keys = (p.kprime + p.bcap == 512) ? 0 : (p.kprime + p.bcap);
  unsigned long long* bars = cbuf + (size_t)QB * qstride + scratch_keys;  // full[stages], empty[stages]
  volatile int* cnt = reinterpret_cast<volatile int*>(bars + 2 * p.stages);        // [QB][2] appended per batch
  volatile float* thr = reinterpret_cast<volatile float*>(const_cast<int*>(cnt) + 2 * QB);
  volatile int* active = reinterpret_cast<volatile int*>(const_cast<float*>(thr) + QB);   // [QB] batch being appended
  volatile int* pending = active + QB;   // [QB] 0 = idle, 1 = batch (1 - active) waits for compaction
  volatile int* frozen = pending + QB;   // [QB] entry count of the batch handed to the compaction warp
  volatile int* nbest = frozen + QB;     // [QB]
  volatile int* done_flag = nbest + QB;  // [1] consumers finished streaming

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int stages = p.stages;
  const uint32_t bar_full0 = smem_u32(bars), bar_empty0 = smem_u32(bars + stages);

  if (tid == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(bar_full0 + 8 * s, 1);
      mbar_init(bar_empty0 + 8 * s, kConsumerWarps);
    }
    mbar_fence_init();
  }
  if (tid < QB) {
    cnt[2 * tid] = 0;
    cnt[2 * tid + 1] = 0;
    thr[tid] = -INFINITY;
    active[tid] = 0;
    pending[tid] = 0;
    frozen[tid] = 0;
    nbest[tid] = 0;
  }
  if (tid == 0) done_flag[0] = 0;
  __syncthreads();

  const int grid = gridDim.x;
  const int my_tiles = ((int)blockIdx.x < p.num_tiles) ? (p.num_tiles - 1 - (int)blockIdx.x) / grid + 1 : 0;
  const uint32_t row_bytes = (uint32_t)p.d_pad * 2u;

  if (warp == kConsumerWarps) {
    // ------------------------------------------------------------ producer warp: one elected lane drives the TMA ring
    if (lane == 0) {
      const uint64_t policy = policy_evict_first();
      const uint32_t tiles_s = smem_u32(tiles);
      for (int i = 0; i < my_tiles; ++i) {
        const int s = i % stages;
        const uint32_t use = (uint32_t)(i / stages);
        if (i >= stages) mbar_wait(bar_empty0 + 8 * s, (use & 1u) ^ 1u);
        const int64_t tile = (int64_t)blockIdx.x + (int64_t)i * grid;
        const uint8_t* src = reinterpret_cast<const uint8_t*>(p.rows) + (size_t)tile * p.tile_bytes;
        mbar_expect_tx(bar_full0 + 8 * s, p.tile_bytes);
        bulk_g2s(tiles_s + (uint32_t)s * p.tile_bytes, src, p.tile_bytes, bar_full0 + 8 * s, policy);
      }
    }
    return;
  }

  if (warp == kConsumerWarps + 1) {
    // ------------------------------------------------------------ compaction warp: folds full batches into best[],
    // publishes the rising threshold, and emits the final sorted top-K' lists.  Never blocks the FMA warps.
    const int T = p.kprime + p.bcap;
    unsigned long long* scratch = cbuf + (size_t)QB * qstride;  // only present when T != 512
    for (;;) {
      const bool fin = done_flag[0] != 0;
      __threadfence_block();
      bool any = false;
      for (int q = 0; q < QB; ++q) {
        if (pending[q]) {
          __threadfence_block();
          unsigned long long* best = cbuf + (size_t)q * qstride;
          const unsigned long long* batch = best + p.kprime + (size_t)(1 - active[q]) * p.bcap;
          const int nb = compact_dispatch(T, best, nbest[q], batch, frozen[q], p.kprime, scratch, lane);
          if (lane == 0) {
            nbest[q] = nb;
            if (nb >= p.kprime) thr[q] = key32_score(best[p.kprime - 1]);
            __threadfence_block();
            pending[q] = 0;
          }
          __syncwarp();
          any = true;
        }
      }
      if (fin && !any) break;
      if (!any) __nanosleep(200);
    }
    // final: fold the batch still being appended, then write the sorted list of every query
    for (int q = 0; q < QB; ++q) {
      unsigned long long* best = cbuf + (size_t)q * qstride;
      const int a = active[q];
      const unsigned long long* batch = best + p.kprime + (size_t)a * p.bcap;
      const int nb = compact_dispatch(T, best, nbest[q], batch, min((int)cnt[2 * q + a], p.bcap), p.kprime, scratch, lane);
      unsigned long long* out = p.cand + ((size_t)q * grid + blockIdx.x) * p.kprime;
      for (int z = lane; z < p.kprime; z += 32) out[z] = z < nb ? best[z] : 0ull;
    }
    return;
  }

  // -------------------------------------------------------------- consumer warps
  // query slices in registers as (even, odd) fp32 pairs: lane owns 16-byte chunk c = lane + 32*j of every row
  unsigned long long qr[QB][NCHUNK][4];
#pragma unroll
  for (int q = 0; q < QB; ++q) {
#pragma unroll
    for (int j = 0; j < NCHUNK; ++j) {
      const int c = lane + 32 * j;
      if (EXACT || c < p.ch) {
        const float4* src = reinterpret_cast<const float4*>(p.q + (size_t)q * p.d_pad + (size_t)c * 8);
        const float4 a = __ldg(src), b = __ldg(src + 1);
        qr[q][j][0] = pack_f2(a.x, a.y);
        qr[q][j][1] = pack_f2(a.z, a.w);
        qr[q][j][2] = pack_f2(b.x, b.y);
        qr[q][j][3] = pack_f2(b.z, b.w);
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) qr[q][j][e] = 0ull;
      }
    }
  }

  const int vi = lane / LPV;          // which (row, query) this lane owns after the reduction
  const int ri = vi / QB, qi = vi % QB;
  const bool leader = (lane % LPV) == 0;
  const int trigger = p.bcap - R;  // a batch is handed over while it still has room for one more tile

  for (int i = 0; i < my_tiles; ++i) {
    const int s = i % stages;
    const uint32_t use = (uint32_t)(i / stages);
    const int64_t tile = (int64_t)blockIdx.x + (int64_t)i * grid;
    const int64_t grow = tile * R + warp * RW + ri;
    mbar_wait(bar_full0 + 8 * s, use & 1u);
    float invn = 0.f;
    if (leader) invn = __ldg(p.inv_norm + grow);  // consumed after the reduction: latency hides under the FMAs

    unsigned long long acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = 0ull;
    const uint8_t* wbase = tiles + (size_t)s * p.tile_bytes + (size_t)(warp * RW) * row_bytes + (size_t)lane * 16;
    // software pipeline at (chunk, row) granularity: the 16 bytes of the next step are in flight while this step is
    // converted and multiplied (one uint4 of look-ahead keeps the register budget under the 200-register ceiling)
    uint4 cur = make_uint4(0u, 0u, 0u, 0u);
    if (EXACT || lane < p.ch) cur = *reinterpret_cast<const uint4*>(wbase);
#pragma unroll
    for (int step = 0; step < NCHUNK * RW; ++step) {
      const int j = step / RW, r = step % RW;
      uint4 nxt = make_uint4(0u, 0u, 0u, 0u);
      if (step + 1 < NCHUNK * RW) {
        const int jn = (step + 1) / RW, rn = (step + 1) % RW;
        if (EXACT || lane + 32 * jn < p.ch)
          nxt = *reinterpret_cast<const uint4*>(wbase + (size_t)rn * row_bytes + (size_t)jn * 512);
      }
      const unsigned long long x0 = h2_to_f2(cur.x), x1 = h2_to_f2(cur.y);
      const unsigned long long x2 = h2_to_f2(cur.z), x3 = h2_to_f2(cur.w);
#pragma unroll
      for (int q = 0; q < QB; ++q) {
        unsigned long long a = acc[r * QB + q];
        a = ffma2(x0, qr[q][j][0], a);
        a = ffma2(x1, qr[q][j][1], a);
        a = ffma2(x2, qr[q][j][2], a);
        a = ffma2(x3, qr[q][j][3], a);
        acc[r * QB + q] = a;
      }
      cur = nxt;
    }
    // all smem reads of this stage are consumed (their values fed the FMAs above) -> release the slot
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_empty0 + 8 * s);

    float part[V];
#pragma unroll
    for (int v = 0; v < V; ++v)
      part[v] = __uint_as_float((uint32_t)(acc[v] & 0xffffffffull)) + __uint_as_float((uint32_t)(acc[v] >> 32));
    const float dot = warp_reduce_multi<V>(part, lane);
    if (leader) {
      const float score = dot * invn;
      if (grow < p.n && score > thr[qi]) {
        const int a = active[qi];
        const int pos = atomicAdd(const_cast<int*>(&cnt[2 * qi + a]), 1);
        if (pos < p.bcap) cbuf[(size_t)qi * qstride + p.kprime + (size_t)a * p.bcap + pos] = make_key32(score, (uint32_t)grow);
      }
    }
    bool need = false;
#pragma unroll
    for (int q = 0; q < QB; ++q) need |= (cnt[2 * q + active[q]] > trigger);
    need = named_bar_or(2, kConsumerThreads, need);
    if (need) {
      // hand the nearly full batch of every such query to the compaction warp and continue on the other batch
      if (tid == 0) {
        for (int q = 0; q < QB; ++q) {
          const int a = active[q];
          const int c = cnt[2 * q + a];
          if (c > trigger) {
            while (pending[q]) __nanosleep(64);  // previous hand-over still being folded (practically never)
            __threadfence_block();
            frozen[q] = min(c, p.bcap);
            cnt[2 * q + (1 - a)] = 0;
            active[q] = 1 - a;
            __threadfence_block();
            pending[q] = 1;
          }
        }
      }
      named_bar_sync(1, kConsumerThreads);
    }
  }

  // -------------------------------------------------------------- streaming finished: the compaction warp finalises
  named_bar_sync(1, kConsumerThreads);
  if (tid == 0) {
    __threadfence_block();
    done_flag[0] = 1;
  }
}

// ------------------------------------------------------------------------------------------------ merge kernel
constexpr int kSelCap = 2048;  // shared-memory capacity of the window (winner) set

struct MergeParams {
  const unsigned long long* cand;  // [nq][G][kprime] sorted descending lists
  int32_t G;
  int32_t kprime;
  int32_t heads_per_list;    // R = ceil(kprime / G)
  int32_t heads_pow2;        // power of two >= G * R  (<= kSelCap)
  const __half* rows;
  const float* q;            // [nq][d_pad] the caller's fp32 queries (exact stage)
  const float* eps;          // [nq] error bound of the approximate scores (0 for an all-zero query)
  int32_t* fallback;         // [nq] raised when the lists cannot serve the window
  int32_t d_pad;
  int32_t ch;
  int64_t id_base;
  int32_t k;
  int64_t* out_ids;          // [nq][k]
  double* out_scores;        // [nq][k]
  int32_t* out_counts;       // [nq]
};

__device__ __forceinline__ void block_sort_desc_u64(unsigned long long* a, int len, int tid, int nt) {
  for (int k = 2; k <= len; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < len; i += nt) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long x = a[i], y = a[ixj];
          const bool desc = (i & k) == 0;
          if (desc ? (x < y) : (x > y)) {
            a[i] = y;
            a[ixj] = x;
          }
        }
      }
      __syncthreads();
    }
  }
}

// One CTA per query.  (1) a lower bound of the global k-th best approximate key = the k-th largest among the first
// R = ceil(K'/G) entries of every list (G*R >= K' >= k real keys); (2) every list contributes its prefix inside the
// error window below that key; a FULL list whose last entry is still inside the window may have dropped members ->
// fallback; (3) exact fp64 re-score of the whole window; (4) final order, emit k.
__global__ void __launch_bounds__(kMergeThreads, 1) dense_merge_kernel(const MergeParams p) {
  extern __shared__ __align__(16) uint8_t msmem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nt = blockDim.x, nw = nt >> 5;
  const int qi = blockIdx.x;
  const int G = p.G, K = p.kprime;
  unsigned long long* sel = reinterpret_cast<unsigned long long*>(msmem);   // [kSelCap]
  unsigned long long* ek = sel + kSelCap;                                   // [kSelCap] exact score keys
  uint32_t* ei = reinterpret_cast<uint32_t*>(ek + kSelCap);                 // [kSelCap] row index
  float* q_s = reinterpret_cast<float*>(ei + kSelCap);                      // [d_pad]   the query, staged once
  __shared__ double qq_s;
  __shared__ int s_nsel, s_trunc;
  __shared__ unsigned long long s_bound;
  const unsigned long long* L = p.cand + (size_t)qi * G * K;

  // (1) bound from the list heads
  const int R = p.heads_per_list, nh = G * R, HP = p.heads_pow2;
  for (int t = tid; t < HP; t += nt) sel[t] = t < nh ? L[(size_t)(t / R) * K + (t % R)] : 0ull;
  if (tid == 0) {
    s_nsel = 0;
    s_trunc = 0;
  }
  __syncthreads();
  block_sort_desc_u64(sel, HP, tid, nt);
  // fewer than k rows in the whole corpus -> sel[k-1] is an empty slot (0): everything is a member
  if (tid == 0) s_bound = sel[p.k - 1] != 0ull ? window_lo_key(sel[p.k - 1], p.eps[qi]) : 0ull;
  __syncthreads();
  const unsigned long long bound = s_bound;
  __syncthreads();  // sel is reused below

  // (2) gather every list's prefix >= bound (lists are sorted descending; empty slots are key 0)
  for (int g = warp; g < G; g += nw) {
    const unsigned long long* lst = L + (size_t)g * K;
    for (int base = 0; base < K; base += 32) {
      const unsigned long long key = lst[base + lane];
      const bool pass = key >= bound && key != 0ull;
      const unsigned m = __ballot_sync(0xffffffffu, pass);
      if (m == 0u) break;
      int pos = 0;
      if (lane == 0) pos = atomicAdd(&s_nsel, __popc(m));
      pos = __shfl_sync(0xffffffffu, pos, 0);
      if (pass) {
        const int at = pos + __popc(m & ((1u << lane) - 1u));
        if (at < kSelCap) sel[at] = key;
      }
      if (m != 0xffffffffu) break;
      if (base + 32 >= K && lane == 0) s_trunc = 1;  // the whole (full) list is inside the window
    }
  }
  __syncthreads();
  const int nsel = s_nsel;
  if (nsel > kSelCap || s_trunc) {
    if (tid == 0) p.fallback[qi] = 1;
    return;
  }
  int P = 32;
  while (P < nsel) P <<= 1;

  RescoreArgs ra;
  ra.rows = p.rows;
  ra.q = p.q + (size_t)qi * p.d_pad;
  ra.d_pad = p.d_pad;
  ra.ch = p.ch;
  ra.id_base = p.id_base;
  ra.k = p.k;
  ra.out_ids = p.out_ids + (size_t)qi * p.k;
  ra.out_scores = p.out_scores + (size_t)qi * p.k;
  ra.out_count = p.out_counts + qi;
  rescore_and_emit(sel, nsel, P, ek, ei, &qq_s, q_s, ra);
}

// ------------------------------------------------------------------------------------------------ query preparation
// One CTA per operand row r (rows >= nq are padding): qn[r] = q[r] / ||q[r]|| in fp32 (the scans rank by cosine, so the
// caller's scale must not reach the fp32 / fp16 arithmetic), optionally q16[r] = fp16(qn[r]) for the tcgen05 scan, and
// eps[r] = the bound on |approximate - exact cosine| the hand-off window uses (0 for an all-zero query).
__global__ void __launch_bounds__(256) dense_prep_queries_kernel(const float* __restrict__ q_pad, int nq, int d_pad,
                                                                 float* __restrict__ qn, __half* __restrict__ q16,
                                                                 float* __restrict__ eps, int mma) {
  __shared__ double s_red[8];
  __shared__ double s_tot;
  const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool real = r < nq;
  const float* src = q_pad + (size_t)r * d_pad;
  double ss = 0.0;
  if (real)
    for (int i = tid; i < d_pad; i += blockDim.x) {
      const double v = (double)src[i];
      ss += v * v;
    }
  for (int o = 16; o; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if (lane == 0) s_red[warp] = ss;
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_red[w];
    s_tot = t;
  }
  __syncthreads();
  const double nrm = sqrt(s_tot);
  const bool zero = !(nrm > 0.0) || !real;
  double dd = 0.0;  // ||fp16(qn) - qn||^2
  for (int i = tid; i < d_pad; i += blockDim.x) {
    const float v = zero ? 0.f : (float)((double)src[i] / nrm);
    if (qn) qn[(size_t)r * d_pad + i] = v;
    if (q16) {
      const __half h = __float2half_rn(v);
      q16[(size_t)r * d_pad + i] = h;
      const double e = (double)__half2float(h) - (double)v;
      dd += e * e;
    }
  }
  if (eps == nullptr || !real) return;
  for (int o = 16; o; o >>= 1) dd += __shfl_xor_sync(0xffffffffu, dd, o);
  __syncthreads();
  if (lane == 0) s_red[warp] = dd;
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_red[w];
    float e = 0.f;
    if (!zero) e = mma ? (float)(sqrt(t) * 1.0001) + dense_eps_mma_acc(d_pad) : dense_eps_fp32(d_pad);
    eps[r] = e;
  }
}

// ------------------------------------------------------------------------------------------------ exact fallback
// One CTA per FLAGGED query (the others exit at once): brute force over every stored row in fp64 -- 1024 rows per round
// are scored by the CTA's 32 warps and folded into the running best list by a 2048-pair bitonic sort (skipped when no
// new row beats the current k-th best).  Slow (tens of ms at 1 M rows) and exact for any score distribution.
constexpr int kFbThreads = 1024;
constexpr int kFbBest = 1024;  // >= the largest supported k

struct FallbackParams {
  const int32_t* flag;   // [nq]
  const __half* rows;
  const float* q;        // [nq][d_pad]
  int64_t n;
  int32_t d_pad, ch;
  int64_t id_base;
  int32_t k;
  int64_t* out_ids;
  double* out_scores;
  int32_t* out_counts;
};

__global__ void __launch_bounds__(kFbThreads, 1) dense_exact_fallback_kernel(const FallbackParams p) {
  const int qi = blockIdx.x;
  if (p.flag[qi] == 0) return;
  __shared__ unsigned long long ek[2 * kFbBest];
  __shared__ uint32_t ei[2 * kFbBest];
  __shared__ double qq_s;
  __shared__ int s_beats;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nt = blockDim.x, nw = nt >> 5;
  const float* q = p.q + (size_t)qi * p.d_pad;
  const double qn = query_norm_cta(q, p.d_pad, &qq_s);
  if (!(qn > 0.0)) {
    // all-zero query: every cosine is exactly 0 -> the first k rows in index order, no scan needed
    const int m = (int)min((int64_t)p.k, p.n);
    for (int i = tid; i < p.k; i += nt) {
      p.out_ids[(size_t)qi * p.k + i] = i < m ? p.id_base + i : -1;
      p.out_scores[(size_t)qi * p.k + i] = 0.0;
    }
    if (tid == 0) p.out_counts[qi] = m;
    return;
  }
  for (int i = tid; i < 2 * kFbBest; i += nt) {
    ek[i] = 0ull;
    ei[i] = 0xffffffffu;
  }
  __syncthreads();
  for (int64_t r0 = 0; r0 < p.n; r0 += kFbBest) {
    if (tid == 0) s_beats = 0;
    __syncthreads();
    const unsigned long long kth = ek[p.k - 1];  // 0 while fewer than k rows have been seen
    bool beat = false;
    for (int c = warp; c < kFbBest; c += nw) {
      const int64_t row = r0 + c;
      unsigned long long okey = 0ull;
      if (row < p.n) {
        okey = f64_orderable(exact_cosine_warp(p.rows, (uint32_t)row, q, p.d_pad, p.ch, qn, lane));
        if (okey == 0ull) okey = 1ull;
      }
      if (lane == 0) {
        ek[kFbBest + c] = okey;
        ei[kFbBest + c] = row < p.n ? (uint32_t)row : 0xffffffffu;
        beat |= okey > kth;   // equal keys: the earlier row is already in the list and wins the tie
      }
    }
    if (beat) s_beats = 1;
    __syncthreads();
    if (s_beats) sort_exact_pairs(ek, ei, 2 * kFbBest, tid, nt);
    __syncthreads();
  }
  RescoreArgs ra;
  ra.rows = p.rows;
  ra.q = q;
  ra.d_pad = p.d_pad;
  ra.ch = p.ch;
  ra.id_base = p.id_base;
  ra.k = p.k;
  ra.out_ids = p.out_ids + (size_t)qi * p.k;
  ra.out_scores = p.out_scores + (size_t)qi * p.k;
  ra.out_count = p.out_counts + qi;
  emit_exact_pairs(ek, ei, kFbBest, ra);
}

// ------------------------------------------------------------------------------------------------ host side
constexpr int kDenseMaxK = 1024;  // per-call top_k limit of both scans (per-CTA lists / winner buffers)

int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

struct ScanPlan {
  int nchunk, rw, qb_max, kprime, bcap, stages, grid, num_tiles;
  uint32_t tile_bytes;
  size_t scan_smem, merge_smem;
  int heads_per_list, heads_pow2;
};

int supported_nchunk(int ch) {
  const int need = (ch + 31) / 32;
  static const int sup[] = {1, 2, 3, 4, 6, 8, 12, 16};
  for (int s : sup)
    if (s >= need) return s;
  return -1;
}

int make_plan(sb_ctx* ctx, const DenseIndex& ix, int k, ScanPlan* pl) {
  const int ch = ix.d_pad / 8;
  pl->nchunk = supported_nchunk(ch);
  SB_REQUIRE(pl->nchunk > 0, SB_ERR_UNSUPPORTED, "dense: dimension %d too large (max 4096)", ix.d);
  pl->rw = pl->nchunk <= 4 ? 4 : (pl->nchunk <= 8 ? 2 : 1);
  pl->qb_max = pl->nchunk <= 4 ? 4 : (pl->nchunk <= 8 ? 2 : 1);
  // per-CTA list length: >= k (the k-th best approximate key must be in the lists); the spare entries above k are what
  // usually lets a list serve the error window without a fallback
  pl->kprime = next_pow2(k + 28);
  if (pl->kprime < 128) pl->kprime = 128;
  if (pl->kprime > kDenseMaxK) pl->kprime = kDenseMaxK;
  SB_REQUIRE(k <= kDenseMaxK, SB_ERR_UNSUPPORTED, "dense: top_k %d too large (max %d per call)", k, kDenseMaxK);
  const int R = kConsumerWarps * pl->rw;
  // compaction sorts best[K'] + one batch in registers across one warp: 512 / 1024 / 1024 / 2048 keys
  pl->bcap = pl->kprime <= 256 ? 3 * pl->kprime : pl->kprime;
  pl->tile_bytes = (uint32_t)R * (uint32_t)ix.d_pad * 2u;
  pl->num_tiles = (int)(ix.n_pad / R);
  const size_t budget = ctx->smem_optin;
  const size_t per_q = (size_t)(pl->kprime + 2 * pl->bcap) * 8;
  const size_t scratch = (pl->kprime + pl->bcap == 512) ? 0 : (size_t)(pl->kprime + pl->bcap) * 8;
  while ((size_t)pl->qb_max * per_q + scratch + 1024 + 2 * (size_t)pl->tile_bytes > budget) {
    if (pl->qb_max > 1) { pl->qb_max >>= 1; continue; }
    sb_set_error("dense: configuration does not fit shared memory (d=%d, k=%d)", ix.d, k);
    return SB_ERR_UNSUPPORTED;
  }
  const size_t fixed = (size_t)pl->qb_max * per_q + scratch;
  int stages = (int)((budget - fixed - 1024) / pl->tile_bytes);
  if (stages > 8) stages = 8;
  if (stages < 2) stages = 2;
  pl->stages = stages;
  pl->scan_smem = (size_t)stages * pl->tile_bytes + fixed + 2 * 8 * (size_t)stages + 256;
  pl->grid = ctx->num_sms < pl->num_tiles ? ctx->num_sms : pl->num_tiles;
  if (pl->grid < 1) pl->grid = 1;
  pl->heads_per_list = (pl->kprime + pl->grid - 1) / pl->grid;
  pl->heads_pow2 = next_pow2(pl->grid * pl->heads_per_list);
  SB_REQUIRE(pl->heads_pow2 <= kSelCap, SB_ERR_UNSUPPORTED, "dense: internal merge capacity exceeded");
  pl->merge_smem = (size_t)kSelCap * 20 + (size_t)ix.d_pad * 4 + 64;
  return SB_OK;
}

template <int NCHUNK, int QB, int RW>
int launch_scan(const ScanParams& sp, const ScanPlan& pl, cudaStream_t st) {
  if (sp.ch == NCHUNK * 32) {
    auto kern = dense_scan_kernel<NCHUNK, QB, RW, true>;
    SB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.scan_smem));
    kern<<<pl.grid, kScanThreads, pl.scan_smem, st>>>(sp);
  } else {
    auto kern = dense_scan_kernel<NCHUNK, QB, RW, false>;
    SB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.scan_smem));
    kern<<<pl.grid, kScanThreads, pl.scan_smem, st>>>(sp);
  }
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

template <int NCHUNK, int RW>
int dispatch_qb(int qb, const ScanParams& sp, const ScanPlan& pl, cudaStream_t st) {
  if constexpr (NCHUNK <= 4) {
    if (qb == 4) return launch_scan<NCHUNK, 4, RW>(sp, pl, st);
  }
  if constexpr (NCHUNK <= 8) {
    if (qb == 2) return launch_scan<NCHUNK, 2, RW>(sp, pl, st);
  }
  return launch_scan<NCHUNK, 1, RW>(sp, pl, st);
}

int dispatch_scan(int qb, const ScanParams& sp, const ScanPlan& pl, cudaStream_t st) {
  switch (pl.nchunk) {
    case 1: return dispatch_qb<1, 4>(qb, sp, pl, st);
    case 2: return dispatch_qb<2, 4>(qb, sp, pl, st);
    case 3: return dispatch_qb<3, 4>(qb, sp, pl, st);
    case 4: return dispatch_qb<4, 4>(qb, sp, pl, st);
    case 6: return dispatch_qb<6, 2>(qb, sp, pl, st);
    case 8: return dispatch_qb<8, 2>(qb, sp, pl, st);
    case 12: return dispatch_qb<12, 1>(qb, sp, pl, st);
    case 16: return dispatch_qb<16, 1>(qb, sp, pl, st);
  }
  sb_set_error("dense: unsupported chunk count %d", pl.nchunk);
  return SB_ERR_UNSUPPORTED;
}

// q_pad: [B][d_pad] fp32 device, zero padded.  Enqueues all scan passes of a chunk of queries, then ONE merge launch
// (one CTA per query) for the whole chunk.
constexpr int kMergeChunk = 256;

int dense_topk_enqueue(sb_ctx* ctx, DenseIndex& ix, const float* q_pad, int B, int k, int64_t* out_ids,
                       double* out_scores, int32_t* out_counts, cudaStream_t st) {
  ScanPlan pl;
  int rc = make_plan(ctx, ix, k, &pl);
  if (rc) return rc;
  // batches of >= 16 queries ride the tensor cores: one HBM pass per 64 / 128 queries instead of one per 4
  if (ctx->dense_mode != 1 && dense_mma_eligible(ctx, ix, B))
    return dense_mma_topk_enqueue(ctx, ix, q_pad, B, k, out_ids, out_scores, out_counts, st);
  const int chunk = B < kMergeChunk ? B : kMergeChunk;
  const size_t per_q = (size_t)pl.grid * pl.kprime;
  rc = ctx->cand_dev.reserve((size_t)chunk * per_q * 8);
  if (rc) return rc;
  // normalised queries for the scan, eps + fallback flags for the hand-off
  float *qn = nullptr, *eps = nullptr;
  int32_t* fb = nullptr;
  if ((rc = dense_prep_queries(ctx, ix, q_pad, B, B, /*mma=*/false, &qn, nullptr, &eps, &fb, st))) return rc;
  SB_CUDA(cudaFuncSetAttribute(dense_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.merge_smem));
  for (int c0 = 0; c0 < B; c0 += chunk) {
    const int nq = std::min(chunk, B - c0);
    int b0 = 0;
    while (b0 < nq) {
      int qb = pl.qb_max;
      while (qb > nq - b0) qb >>= 1;
      ScanParams sp;
      sp.rows = ix.rows;
      sp.inv_norm = ix.inv_norm;
      sp.q = qn + (size_t)(c0 + b0) * ix.d_pad;
      sp.cand = ctx->cand_dev.as<unsigned long long>() + (size_t)b0 * per_q;
      sp.n = ix.n;
      sp.d_pad = ix.d_pad;
      sp.ch = ix.d_pad / 8;
      sp.num_tiles = pl.num_tiles;
      sp.kprime = pl.kprime;
      sp.bcap = pl.bcap;
      sp.stages = pl.stages;
      sp.tile_bytes = pl.tile_bytes;
      {
        ProfScope ps(ctx, SB_PROF_DENSE_SCAN, st);
        rc = dispatch_scan(qb, sp, pl, st);
      }
      if (rc) return rc;
      b0 += qb;
    }
    MergeParams mp;
    mp.cand = ctx->cand_dev.as<unsigned long long>();
    mp.G = pl.grid;
    mp.kprime = pl.kprime;
    mp.heads_per_list = pl.heads_per_list;
    mp.heads_pow2 = pl.heads_pow2;
    mp.rows = ix.rows;
    mp.q = q_pad + (size_t)c0 * ix.d_pad;
    mp.eps = eps + c0;
    mp.fallback = fb + c0;
    mp.d_pad = ix.d_pad;
    mp.ch = ix.d_pad / 8;
    mp.id_base = ix.id_base;
    mp.k = k;
    mp.out_ids = out_ids + (size_t)c0 * k;
    mp.out_scores = out_scores + (size_t)c0 * k;
    mp.out_counts = out_counts + c0;
    {
      ProfScope ps(ctx, SB_PROF_DENSE_MERGE, st);
      dense_merge_kernel<<<nq, kMergeThreads, pl.merge_smem, st>>>(mp);
    }
    SB_CUDA(cudaGetLastError());
  }
  return dense_fallback_enqueue(ctx, ix, q_pad, B, k, fb, out_ids, out_scores, out_counts, st);
}

__global__ void fill_empty_topk_kernel(int64_t* ids, double* sc, int32_t* cnt, int B, int k) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B * k) {
    ids[i] = -1;
    sc[i] = 0.0;
  }
  if (i < B) cnt[i] = 0;
}

__global__ void dense_fetch_kernel(const __half* rows, int d, int d_pad, int64_t n, int64_t id_base,
                                   const int64_t* ids, int n_ids, float* out) {
  int r = blockIdx.x;
  if (r >= n_ids) return;
  int64_t idx = ids[r] - id_base;
  for (int i = threadIdx.x; i < d; i += blockDim.x)
    out[(size_t)r * d + i] = (idx >= 0 && idx < n) ? __half2float(rows[(size_t)idx * d_pad + i]) : 0.f;
}

}  // namespace

// Shared with dense_mma.cu: query preparation (normalised fp32 copy, optional fp16 operand rows, eps, cleared fallback
// flags) and the brute-force fallback launch.  `rows` >= B operand rows are prepared (rows >= B are zero padding).
int dense_prep_queries(sb_ctx* ctx, const DenseIndex& ix, const float* q_pad, int B, int rows, bool mma, float** qn_out,
                       __half* q16, float** eps_out, int32_t** fb_out, cudaStream_t st) {
  int rc;
  if ((rc = ctx->qaux_dev.reserve((size_t)rows * 8 + 64))) return rc;
  float* eps = ctx->qaux_dev.as<float>();
  int32_t* fb = reinterpret_cast<int32_t*>(eps + rows);
  float* qn = nullptr;
  if (qn_out) {
    if ((rc = ctx->qn_dev.reserve((size_t)rows * ix.d_pad * sizeof(float)))) return rc;
    qn = ctx->qn_dev.as<float>();
    *qn_out = qn;
  }
  SB_CUDA(cudaMemsetAsync(fb, 0, (size_t)rows * 4, st));
  ctx->launches += 1;
  dense_prep_queries_kernel<<<rows, 256, 0, st>>>(q_pad, B, ix.d_pad, qn, q16, eps, mma ? 1 : 0);
  SB_CUDA(cudaGetLastError());
  *eps_out = eps;
  *fb_out = fb;
  return SB_OK;
}

int dense_fallback_enqueue(sb_ctx* ctx, const DenseIndex& ix, const float* q_pad, int B, int k, const int32_t* fb,
                           int64_t* out_ids, double* out_scores, int32_t* out_counts, cudaStream_t st) {
  FallbackParams fp;
  fp.flag = fb;
  fp.rows = ix.rows;
  fp.q = q_pad;
  fp.n = ix.n;
  fp.d_pad = ix.d_pad;
  fp.ch = ix.d_pad / 8;
  fp.id_base = ix.id_base;
  fp.k = k;
  fp.out_ids = out_ids;
  fp.out_scores = out_scores;
  fp.out_counts = out_counts;
  ctx->launches += 1;
  dense_exact_fallback_kernel<<<B, kFbThreads, 0, st>>>(fp);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

// Shared with other translation units (hybrid batch path, scorers).
int sb_dense_pad_queries(sb_ctx* ctx, const DenseIndex& ix, const float* q, int B, bool q_on_device, float** q_pad_out,
                         cudaStream_t st) {
  int rc = ctx->q_dev.reserve((size_t)B * ix.d_pad * sizeof(float));
  if (rc) return rc;
  float* qp = ctx->q_dev.as<float>();
  if (ix.d_pad != ix.d) SB_CUDA(cudaMemsetAsync(qp, 0, (size_t)B * ix.d_pad * sizeof(float), st));
  SB_CUDA(cudaMemcpy2DAsync(qp, (size_t)ix.d_pad * sizeof(float), q, (size_t)ix.d * sizeof(float),
                            (size_t)ix.d * sizeof(float), (size_t)B,
                            q_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  *q_pad_out = qp;
  return SB_OK;
}

extern "C" {

int sb_dense_load(sb_ctx* ctx, int slot, const void* vecs, int64_t n, int32_t d, int32_t dtype, int64_t id_base) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_dense_load: ctx is NULL");
  SB_REQUIRE(slot >= 0 && slot < SB_MAX_DENSE_SLOTS, SB_ERR_ARG, "sb_dense_load: bad slot %d", slot);
  SB_REQUIRE(n >= 0 && d > 0 && d <= 4096, SB_ERR_ARG, "sb_dense_load: bad shape n=%lld d=%d", (long long)n, d);
  SB_REQUIRE(n < (1ll << 31), SB_ERR_ARG, "sb_dense_load: a shard holds at most 2^31-1 rows");
  SB_REQUIRE(dtype == SB_F32 || dtype == SB_F16, SB_ERR_ARG, "sb_dense_load: dtype must be SB_F32 or SB_F16");
  SB_REQUIRE(n == 0 || vecs != nullptr, SB_ERR_ARG, "sb_dense_load: vecs is NULL");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  DenseIndex& ix = ctx->dense[slot];
  SB_CUDA(cudaStreamSynchronize(ctx->stream));
  if (ix.rows) cudaFree(ix.rows);
  if (ix.inv_norm) cudaFree(ix.inv_norm);
  ix = DenseIndex();
  ix.n = n;
  ix.d = d;
  ix.d_pad = (d + 7) / 8 * 8;
  ix.n_pad = (n + kRowPad - 1) / kRowPad * kRowPad;
  ix.id_base = id_base;
  if (n == 0) return SB_OK;
  SB_CUDA(cudaMalloc(&ix.rows, (size_t)ix.n_pad * ix.d_pad * sizeof(__half)));
  SB_CUDA(cudaMalloc(&ix.inv_norm, (size_t)ix.n_pad * sizeof(float)));
  SB_CUDA(cudaMemsetAsync(ix.rows, 0, (size_t)ix.n_pad * ix.d_pad * sizeof(__half), ctx->stream));
  SB_CUDA(cudaMemsetAsync(ix.inv_norm, 0, (size_t)ix.n_pad * sizeof(float), ctx->stream));
  // staged upload: chunks of rows through a device staging buffer
  const size_t esz = dtype == SB_F32 ? 4 : 2;
  const int64_t chunk_rows = std::max<int64_t>(1, (int64_t)((256ull << 20) / ((size_t)d * esz)));
  int rc = ctx->misc_dev.reserve((size_t)std::min<int64_t>(chunk_rows, n) * d * esz);
  if (rc) return rc;
  for (int64_t r0 = 0; r0 < n; r0 += chunk_rows) {
    const int64_t nr = std::min<int64_t>(chunk_rows, n - r0);
    const uint8_t* src = reinterpret_cast<const uint8_t*>(vecs) + (size_t)r0 * d * esz;
    SB_CUDA(cudaMemcpyAsync(ctx->misc_dev.p, src, (size_t)nr * d * esz, cudaMemcpyHostToDevice, ctx->stream));
    const int wpb = 8;
    const unsigned blocks = (unsigned)((nr + wpb - 1) / wpb);
    if (dtype == SB_F32)
      dense_store_rows_kernel<float><<<blocks, wpb * 32, 0, ctx->stream>>>(ctx->misc_dev.as<float>(), nr, d, ix.d_pad,
                                                                           ix.rows, ix.inv_norm, r0, true);
    else
      dense_store_rows_kernel<__half><<<blocks, wpb * 32, 0, ctx->stream>>>(ctx->misc_dev.as<__half>(), nr, d,
                                                                            ix.d_pad, ix.rows, ix.inv_norm, r0, false);
    SB_CUDA(cudaGetLastError());
    SB_CUDA(cudaStreamSynchronize(ctx->stream));  // staging buffer is reused by the next chunk
  }
  return SB_OK;
}

int sb_dense_set_mode(sb_ctx* ctx, int mode) {
  SB_REQUIRE(ctx != nullptr && (mode == 0 || mode == 1), SB_ERR_ARG, "sb_dense_set_mode: bad arguments");
  std::lock_guard<std::mutex> lk(ctx->mu);
  ctx->dense_mode = mode;
  return SB_OK;
}

int64_t sb_dense_count(sb_ctx* ctx, int slot) {
  if (!ctx || slot < 0 || slot >= SB_MAX_DENSE_SLOTS) return -1;
  return ctx->dense[slot].n;
}

int32_t sb_dense_dim(sb_ctx* ctx, int slot) {
  if (!ctx || slot < 0 || slot >= SB_MAX_DENSE_SLOTS) return -1;
  return ctx->dense[slot].d;
}

int sb_dense_topk_dev(sb_ctx* ctx, int slot, const float* q_dev, int32_t B, int32_t k, int64_t* out_ids_dev,
                      double* out_scores_dev, int32_t* out_counts_dev, void* stream) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_dense_topk_dev: ctx is NULL");
  SB_REQUIRE(slot >= 0 && slot < SB_MAX_DENSE_SLOTS, SB_ERR_ARG, "sb_dense_topk_dev: bad slot %d", slot);
  SB_REQUIRE(B >= 0 && k > 0, SB_ERR_ARG, "sb_dense_topk_dev: bad B=%d k=%d", B, k);
  if (B == 0) return SB_OK;
  SB_REQUIRE(q_dev && out_ids_dev && out_scores_dev && out_counts_dev, SB_ERR_ARG, "sb_dense_topk_dev: NULL buffer");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  cudaStream_t st = pick_stream(ctx, stream);
  DenseIndex& ix = ctx->dense[slot];
  SB_REQUIRE(ix.d > 0, SB_ERR_STATE, "sb_dense_topk: dense slot %d has no index loaded", slot);
  if (ix.n == 0) {
    fill_empty_topk_kernel<<<(B * k + 255) / 256, 256, 0, st>>>(out_ids_dev, out_scores_dev, out_counts_dev, B, k);
    SB_CUDA(cudaGetLastError());
    return SB_OK;
  }
  float* q_pad = nullptr;
  int rc = sb_dense_pad_queries(ctx, ix, q_dev, B, true, &q_pad, st);
  if (rc) return rc;
  return dense_topk_enqueue(ctx, ix, q_pad, B, k, out_ids_dev, out_scores_dev, out_counts_dev, st);
}

int sb_dense_topk(sb_ctx* ctx, int slot, const float* q, int32_t B, int32_t k, int64_t* out_ids, double* out_scores,
                  int32_t* out_counts) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_dense_topk: ctx is NULL");
  SB_REQUIRE(slot >= 0 && slot < SB_MAX_DENSE_SLOTS, SB_ERR_ARG, "sb_dense_topk: bad slot %d", slot);
  SB_REQUIRE(B >= 0 && k > 0, SB_ERR_ARG, "sb_dense_topk: bad B=%d k=%d", B, k);
  if (B == 0) return SB_OK;
  SB_REQUIRE(q && out_ids && out_scores && out_counts, SB_ERR_ARG, "sb_dense_topk: NULL buffer");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  cudaStream_t st = ctx->stream;
  DenseIndex& ix = ctx->dense[slot];
  SB_REQUIRE(ix.d > 0, SB_ERR_STATE, "sb_dense_topk: dense slot %d has no index loaded", slot);
  if (ix.n == 0) {
    for (int i = 0; i < B * k; ++i) { out_ids[i] = -1; out_scores[i] = 0.0; }
    for (int i = 0; i < B; ++i) out_counts[i] = 0;
    return SB_OK;
  }
  int rc;
  const size_t qbytes = (size_t)B * ix.d * sizeof(float);
  const size_t nid = (size_t)B * k;
  // page-locked caller buffers are used in place; pageable ones go through the context's pinned staging
  const bool in_pinned = host_ptr_is_pinned(q);
  const bool out_pinned = host_ptr_is_pinned(out_ids) && host_ptr_is_pinned(out_scores) && host_ptr_is_pinned(out_counts);
  const float* q_src = q;
  if (!in_pinned) {
    if ((rc = ctx->pin_in.reserve(qbytes))) return rc;
    memcpy(ctx->pin_in.p, q, qbytes);
    q_src = ctx->pin_in.as<float>();
  }
  float* q_pad = nullptr;
  if ((rc = sb_dense_pad_queries(ctx, ix, q_src, B, false, &q_pad, st))) return rc;
  if ((rc = ctx->out_ids_dev.reserve(nid * 8))) return rc;
  if ((rc = ctx->out_sc_dev.reserve(nid * 8))) return rc;
  if ((rc = ctx->out_cnt_dev.reserve((size_t)B * 4))) return rc;
  if ((rc = dense_topk_enqueue(ctx, ix, q_pad, B, k, ctx->out_ids_dev.as<int64_t>(), ctx->out_sc_dev.as<double>(),
                               ctx->out_cnt_dev.as<int32_t>(), st)))
    return rc;
  if (out_pinned) {
    SB_CUDA(cudaMemcpyAsync(out_ids, ctx->out_ids_dev.p, nid * 8, cudaMemcpyDeviceToHost, st));
    SB_CUDA(cudaMemcpyAsync(out_scores, ctx->out_sc_dev.p, nid * 8, cudaMemcpyDeviceToHost, st));
    SB_CUDA(cudaMemcpyAsync(out_counts, ctx->out_cnt_dev.p, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    SB_CUDA(cudaStreamSynchronize(st));
    return SB_OK;
  }
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

int sb_dense_fetch(sb_ctx* ctx, int slot, const int64_t* ids, int32_t n_ids, float* out) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_dense_fetch: ctx is NULL");
  SB_REQUIRE(slot >= 0 && slot < SB_MAX_DENSE_SLOTS, SB_ERR_ARG, "sb_dense_fetch: bad slot %d", slot);
  if (n_ids <= 0) return SB_OK;
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  const DenseIndex& ix = ctx->dense[slot];
  SB_REQUIRE(ix.d > 0 && ix.n > 0, SB_ERR_STATE, "sb_dense_fetch: dense slot %d is empty", slot);
  int rc;
  if ((rc = ctx->misc2_dev.reserve((size_t)n_ids * 8))) return rc;
  if ((rc = ctx->misc3_dev.reserve((size_t)n_ids * ix.d * 4))) return rc;
  SB_CUDA(cudaMemcpyAsync(ctx->misc2_dev.p, ids, (size_t)n_ids * 8, cudaMemcpyHostToDevice, ctx->stream));
  dense_fetch_kernel<<<n_ids, 128, 0, ctx->stream>>>(ix.rows, ix.d, ix.d_pad, ix.n, ix.id_base,
                                                     ctx->misc2_dev.as<int64_t>(), n_ids, ctx->misc3_dev.as<float>());
  SB_CUDA(cudaGetLastError());
  SB_CUDA(cudaMemcpyAsync(out, ctx->misc3_dev.p, (size_t)n_ids * ix.d * 4, cudaMemcpyDeviceToHost, ctx->stream));
  SB_CUDA(cudaStreamSynchronize(ctx->stream));
  return SB_OK;
}

}  // extern "C"
