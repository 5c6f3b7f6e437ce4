// dense_mma.cu -- K1b: batched-query dense scan on the 5th-gen tensor cores (tcgen05 / TMEM / TMA).
//
// One HBM pass over the fp16 corpus serves a whole GROUP of queries: the scores of a 128-row corpus tile against all
// queries of the group are one UMMA accumulator  D[128, N] = A[128, D] * Q[N, D]^T  (A = corpus tile, K-major fp16,
// streamed by TMA in 64-column SWIZZLE_128B boxes; B = the normalised fp16 query block, K-major, resident in shared
// memory for the whole kernel; D in tensor memory, double buffered).
//   * dense_scan_mma_kernel<QBN>   one CTA per SM, N = QBN = 16 / 32 / 64 queries (cta_group::1).
//   * dense_scan_mma2_kernel<128>  a CTA PAIR (2-CTA cluster, cta_group::2): one UMMA of M = 256 (128 corpus rows per
//     CTA) x N = 128 queries whose B operand is split across the pair -- each CTA keeps 64 query rows (128 KB at
//     d = 1024, the shared-memory limit of one SM), streams its own A tiles, and receives D[128 rows, 128 queries] in its
//     own tensor memory: 128 queries per HBM pass with no extra L2 traffic.
// The pass stays HBM bound: per 16 KB of corpus the tensor pipe needs 4 MMAs, a third of its capacity at N = 128.
//
// Exactness (dense_common.cuh, DESIGN.md "K1: exactness"):
//   * queries are L2-normalised before the fp16 rounding (cosine is scale invariant; the caller's scale never reaches
//     the fp16 range) and eps[q] = ||fp16(qn) - qn|| + accumulation bound is computed per query;
//   * a sampling pass gives every query a SAFE threshold: (k-th best approximate score of a corpus sample) - 2 eps is
//     <= (global k-th best) - 2 eps, the lower edge of the hand-off window, so every window member survives the epilogue;
//   * survivors are appended to per-(CTA, query) lists; a list that overflows its capacity raises the query's fallback
//     flag instead of dropping anything silently;
//   * dense_select_kernel finds the k-th best approximate key (radix select), gathers EVERY survivor inside the window
//     below it and re-scores them all in fp64 against the stored rows and the caller's fp32 query; a window larger than
//     the winner buffer raises the fallback flag (dense_exact_fallback_kernel, dense.cu).
//
// Warp roles (192 threads, 1 CTA / SM, persistent): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2..5 = epilogue (tcgen05.ld 32x32b, one corpus row per thread).
#include <cuda.h>

#include <math.h>

#include <algorithm>
#include <vector>

#include "dense_common.cuh"
#include "dense_mma.cuh"

namespace {

constexpr int kTileRows = 128;
constexpr int kBK = 64;                       // fp16 elements per 128-byte swizzle row
constexpr uint32_t kATileBytes = kTileRows * kBK * 2;   // 16 KB
constexpr int kMmaThreads = 192;
constexpr int kMaxStages = 8;                 // cap on the TMA ring depth of the scan kernels
constexpr int kSampleTilesPerCta = 2;         // least corpus tiles per CTA of the sampling pass
constexpr int kSelectThreads = 512;
constexpr int kSelStage = 8192;               // survivors staged in shared memory by dense_select_kernel (64 KB)
constexpr int kSelTop = 2048;                 // window (winner) buffer; larger windows go to the exact fallback

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
      "l"(map), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}

__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
  d |= (uint64_t)1 << 16;             // LBO (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;   // SBO: 8 rows x 128 B
  d |= (uint64_t)1 << 46;             // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;             // SWIZZLE_128B
  return d;
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// ---- cta_group::2 forms (the pair kernel); PTX as in cute/arch/{copy_sm100_tma,mma_sm100_umma}.hpp, cutlass/arch/barrier.h
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// shared::cluster address of `smem_addr` (a shared::cta address of this CTA) inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  __syncwarp();
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose completion bytes are signalled on an mbarrier of the LEADER CTA (bar_cluster = mapa(bar, 0))
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar_cluster) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
      "l"(map), "r"(c0), "r"(c1), "r"(bar_cluster)
      : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
// arrive (once all MMAs issued so far have completed) on the barrier at this shared-memory offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"((uint16_t)3)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster) {
  // default semantics (release at CTA scope), as CUTLASS's ClusterBarrier::arrive(cta_id): the tcgen05 fences order the
  // tensor-memory reads; a cluster-scope release would add a full memory barrier per tile (8.5 % of the stall samples)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}

template <int N>
struct TmemLd;
template <>
struct TmemLd<16> {
  static __device__ __forceinline__ void ld(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
  }
};

// Sampling-pass epilogue.  The threshold only needs a LOWER bound of the k-th best score, and the k-th largest of ANY
// set of distinct rows' scores is one: each warp contributes the best score among its 32 rows (one REDUX per query
// column, no atomics, one 8-byte store per (warp, query) at slot `slot` of the CTA's list) instead of all 32.
template <int NV>
__device__ __forceinline__ void sample_emit(const uint32_t (&v)[NV], bool live, float invn, unsigned long long* my_cand,
                                            size_t q_stride, int c0, int slot, int lane) {
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const float score = live ? __uint_as_float(v[j]) * invn : -INFINITY;
    const uint32_t best = __reduce_max_sync(0xffffffffu, f32_orderable(score));
    if (lane == (j & 31)) my_cand[(size_t)(c0 + j) * q_stride + slot] = ((unsigned long long)best << 32) | 0xffffffffull;
  }
}

struct MmaScanParams {
  const float* inv_norm;
  const float* thr_init;        // [QBN] safe initial thresholds (NULL = -inf: sampling pass)
  unsigned long long* cand;     // [QBN][grid][capg]
  int32_t* counts;              // [QBN][grid]
  int32_t* fallback;            // [QBN] raised when a (CTA, query) list overflows capg (NULL: cannot overflow)
  int64_t n;                    // valid rows
  int32_t kb_count;             // d_pad / 64
  int32_t num_tiles;            // tiles visited by this launch
  int32_t tile_first, tile_step; // global tile index = tile_first + t * tile_step,  t in [0, num_tiles)
  int32_t capg;
  int32_t stages;
  // pair kernel, SAMPLING pass only: n_groups query groups of 128 operand rows handled by one launch, one after the other
  // (group g: operand rows [128 g, 128 g + 128) of tm_q, lists at cand + g * group_cand_stride, counts + g * group_cnt_stride)
  int32_t n_groups;
  int64_t group_cand_stride;
  int64_t group_cnt_stride;
};

template <int QBN>
__global__ void __launch_bounds__(kMmaThreads, 1)
dense_scan_mma_kernel(const __grid_constant__ CUtensorMap tm_rows, const __grid_constant__ CUtensorMap tm_q,
                      const MmaScanParams p) {
  extern __shared__ uint8_t msm_raw[];
  const uint32_t raw = smem_u32(msm_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;  // SWIZZLE_128B operands need 1024-byte alignment
  uint8_t* sm = msm_raw + (base - raw);
  constexpr uint32_t kQBlockBytes = QBN * kBK * 2;      // one 64-column block of the query operand
  const uint32_t q_bytes = (uint32_t)p.kb_count * kQBlockBytes;
  const uint32_t a0 = base + q_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + q_bytes + (size_t)p.stages * kATileBytes);
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + p.stages);
  const uint32_t bar_q = smem_u32(bars + 2 * p.stages);
  const uint32_t bar_acc_full = smem_u32(bars + 2 * p.stages + 1), bar_acc_empty = smem_u32(bars + 2 * p.stages + 3);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * p.stages + 6);   // its own 16-byte slot (tcgen05.alloc writes it)
  volatile float* thr = reinterpret_cast<volatile float*>(tmem_slot + 2);   // [QBN]
  int* cnt = reinterpret_cast<int*>(const_cast<float*>(thr) + QBN);        // [QBN]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int grid = gridDim.x, cta = blockIdx.x;
  const int my_tiles = cta < p.num_tiles ? (p.num_tiles - 1 - cta) / grid + 1 : 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_q, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar_acc_full + 8 * s, 1);
      mbar_init(bar_acc_empty + 8 * s, 4);  // one arrival per epilogue warp
    }
    mbar_fence_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_rows) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_q) : "memory");
  }
  for (int i = threadIdx.x; i < QBN; i += blockDim.x) {
    thr[i] = p.thr_init ? p.thr_init[i] : -INFINITY;
    cnt[i] = 0;
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(2 * QBN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer
    if (lane == 0) {
      mbar_expect_tx(bar_q, q_bytes);
      for (int kb = 0; kb < p.kb_count; ++kb) tma_load_2d(base + (uint32_t)kb * kQBlockBytes, &tm_q, kb * kBK, 0, bar_q);
      int it = 0;
      for (int t = 0; t < my_tiles; ++t) {
        const int tile = p.tile_first + (cta + t * grid) * p.tile_step;
        for (int kb = 0; kb < p.kb_count; ++kb, ++it) {
          const int s = it % p.stages;
          const uint32_t use = (uint32_t)(it / p.stages);
          if (it >= p.stages) mbar_wait(bar_empty + 8 * s, (use & 1u) ^ 1u);
          mbar_expect_tx(bar_full + 8 * s, kATileBytes);
          tma_load_2d(a0 + (uint32_t)s * kATileBytes, &tm_rows, kb * kBK, tile * kTileRows, bar_full + 8 * s);
        }
      }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer
    if (lane == 0) {
      // kind::f16: D = f32, A = B = f16 K-major, N >> 3 at [17,23), M >> 4 at [24,29)
      const uint32_t idesc = (1u << 4) | ((uint32_t)(QBN >> 3) << 17) | ((uint32_t)(kTileRows >> 4) << 24);
      mbar_wait(bar_q, 0);
      int it = 0;
      for (int t = 0; t < my_tiles; ++t) {
        const int as = t & 1;
        if (t >= 2) mbar_wait(bar_acc_empty + 8 * as, (((uint32_t)t >> 1) & 1u) ^ 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * QBN);
        for (int kb = 0; kb < p.kb_count; ++kb, ++it) {
          const int s = it % p.stages;
          const uint32_t use = (uint32_t)(it / p.stages);
          mbar_wait(bar_full + 8 * s, use & 1u);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint64_t da = make_smem_desc_sw128(a0 + (uint32_t)s * kATileBytes);
          const uint64_t db = make_smem_desc_sw128(base + (uint32_t)kb * kQBlockBytes);
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k)
            umma_f16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) ? 1u : 0u);
          umma_commit(bar_empty + 8 * s);
        }
        umma_commit(bar_acc_full + 8 * as);
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue warps 2..5: one corpus row per thread
    const int quad = warp & 3;
    unsigned long long* my_cand = p.cand + (size_t)cta * p.capg;
    const size_t q_stride = (size_t)grid * p.capg;
    for (int t = 0; t < my_tiles; ++t) {
      const int as = t & 1;
      const int tile = p.tile_first + (cta + t * grid) * p.tile_step;
      const int64_t row = (int64_t)tile * kTileRows + quad * 32 + lane;
      const float invn = row < p.n ? __ldg(p.inv_norm + row) : 0.f;
      mbar_wait(bar_acc_full + 8 * as, ((uint32_t)t >> 1) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
      for (int c0 = 0; c0 < QBN; c0 += 16) {
        uint32_t v[16];
        TmemLd<16>::ld(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * QBN + c0), v);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (p.thr_init == nullptr) {
          // sampling pass: one key per (warp, query) = the best score among the warp's 32 rows (see sample_emit)
          sample_emit<16>(v, row < p.n, invn, my_cand, q_stride, c0, t * 4 + quad, lane);
          continue;
        }
        if (row < p.n) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float score = __uint_as_float(v[j]) * invn;
            if (score >= thr[c0 + j]) {
              const int pos = atomicAdd(&cnt[c0 + j], 1);
              if (pos < p.capg) my_cand[(size_t)(c0 + j) * q_stride + pos] = make_key32(score, (uint32_t)row);
            }
          }
        }
      }
      // the accumulator stage has been read into registers by this warp -> give it back to the MMA issuer
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty + 8 * as);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  for (int i = threadIdx.x; i < QBN; i += blockDim.x) {
    const int c = p.thr_init == nullptr ? my_tiles * 4 : cnt[i];   // sampling pass: 4 warp maxima per tile
    p.counts[(size_t)i * grid + cta] = min(c, p.capg);
    if (c > p.capg && p.fallback) p.fallback[i] = 1;   // nothing is dropped silently: brute force answers this query
  }
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(2 * QBN) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------ pair kernel
// cta_group::2: CTA rank 0 (the leader) issues every MMA for the pair; both CTAs stream their own A tiles and load
// their own half of the query block, with TMA completion bytes landing on the LEADER's full barriers; tcgen05.commit
// multicasts the "stage free" / "accumulator ready" arrivals to both CTAs; the epilogue warps of both CTAs arrive on the
// leader's "accumulator drained" barrier through the cluster address space.
template <int NQ>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kMmaThreads, 1)
dense_scan_mma2_kernel(const __grid_constant__ CUtensorMap tm_rows, const __grid_constant__ CUtensorMap tm_q,
                       const MmaScanParams p) {
  constexpr int HQ = NQ / 2;                            // operand rows held by each CTA
  extern __shared__ uint8_t msm_raw[];
  const uint32_t raw = smem_u32(msm_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* sm = msm_raw + (base - raw);
  constexpr uint32_t kQBlockBytes = HQ * kBK * 2;
  const uint32_t q_bytes = (uint32_t)p.kb_count * kQBlockBytes;
  const uint32_t a0 = base + q_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + q_bytes + (size_t)p.stages * kATileBytes);
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + p.stages);
  const uint32_t bar_q = smem_u32(bars + 2 * p.stages);
  const uint32_t bar_acc_full = smem_u32(bars + 2 * p.stages + 1), bar_acc_empty = smem_u32(bars + 2 * p.stages + 3);
  const uint32_t bar_qfree = smem_u32(bars + 2 * p.stages + 5);   // every MMA of a query group has completed (both CTAs)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * p.stages + 8);   // its own 16-byte slot (tcgen05.alloc writes it)
  volatile float* thr = reinterpret_cast<volatile float*>(tmem_slot + 2);   // [NQ]
  int* cnt = reinterpret_cast<int*>(const_cast<float*>(thr) + NQ);         // [NQ]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int n_groups = p.thr_init == nullptr ? max(p.n_groups, 1) : 1;   // several groups per launch: sampling pass only
  const int grid = gridDim.x, cta = blockIdx.x;
  const int pair = cta >> 1, npairs = grid >> 1;
  const int n_tp = (p.num_tiles + 1) >> 1;              // tile pairs of this launch
  const int my_tiles = pair < n_tp ? (n_tp - 1 - pair) / npairs + 1 : 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(bar_full + 8 * s, 1);    // used in the leader only: its own expect_tx arrival + the bytes of both CTAs
      mbar_init(bar_empty + 8 * s, 1);   // one multicast commit per use
    }
    mbar_init(bar_q, 1);
    mbar_init(bar_qfree, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar_acc_full + 8 * s, 1);
      mbar_init(bar_acc_empty + 8 * s, 8);  // leader only: 4 epilogue warps x 2 CTAs
    }
    mbar_fence_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_rows) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_q) : "memory");
  }
  for (int i = threadIdx.x; i < NQ; i += blockDim.x) {
    thr[i] = p.thr_init ? p.thr_init[i] : -INFINITY;
    cnt[i] = 0;
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(2 * NQ)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();   // the peer's barriers are initialised before anything is signalled across the pair
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ---------------------------------------------------------------- TMA producer (both CTAs)
    if (lane == 0) {
      const uint32_t lead_q = mapa_u32(bar_q, 0);
      int it = 0;
      for (int g = 0; g < n_groups; ++g) {
      // the query operand of group g replaces that of group g - 1 once every MMA that read it has completed
      if (g > 0) mbar_wait(bar_qfree, (uint32_t)(g - 1) & 1u);
      if (rank == 0) mbar_expect_tx(bar_q, 2u * q_bytes);
      for (int kb = 0; kb < p.kb_count; ++kb)
        tma_load_2d_pair(base + (uint32_t)kb * kQBlockBytes, &tm_q, kb * kBK, g * NQ + (int)rank * HQ, lead_q);
      for (int t = 0; t < my_tiles; ++t) {
        const int li = 2 * (pair + t * npairs) + (int)rank;
        // the odd tile of the last pair may not exist: load tile 0 again (served by L2), the epilogue ignores it
        const int tile = li < p.num_tiles ? p.tile_first + li * p.tile_step : p.tile_first;
        for (int kb = 0; kb < p.kb_count; ++kb, ++it) {
          const int s = it % p.stages;
          const uint32_t use = (uint32_t)(it / p.stages);
          if (it >= p.stages) mbar_wait(bar_empty + 8 * s, (use & 1u) ^ 1u);
          if (rank == 0) mbar_expect_tx(bar_full + 8 * s, 2u * kATileBytes);
          tma_load_2d_pair(a0 + (uint32_t)s * kATileBytes, &tm_rows, kb * kBK, tile * kTileRows,
                           mapa_u32(bar_full + 8 * s, 0));
        }
      }
      }
    }
  } else if (warp == 1) {
    // ---------------------------------------------------------------- MMA issuer (leader CTA only)
    if (lane == 0 && rank == 0) {
      // kind::f16: D = f32, A = B = f16 K-major, N >> 3 at [17,23), M >> 4 at [24,29); M = 256 across the pair
      const uint32_t idesc = (1u << 4) | ((uint32_t)(NQ >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      int it = 0, tt = 0;   // ring slot counter / accumulator-stage counter, both running across the query groups
      for (int g = 0; g < n_groups; ++g) {
      mbar_wait(bar_q, (uint32_t)g & 1u);
      for (int t = 0; t < my_tiles; ++t, ++tt) {
        const int as = tt & 1;
        if (tt >= 2) mbar_wait(bar_acc_empty + 8 * as, (((uint32_t)tt >> 1) & 1u) ^ 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * NQ);
        for (int kb = 0; kb < p.kb_count; ++kb, ++it) {
          const int s = it % p.stages;
          const uint32_t use = (uint32_t)(it / p.stages);
          mbar_wait(bar_full + 8 * s, use & 1u);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint64_t da = make_smem_desc_sw128(a0 + (uint32_t)s * kATileBytes);
          const uint64_t db = make_smem_desc_sw128(base + (uint32_t)kb * kQBlockBytes);
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k)
            umma_f16_pair(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) ? 1u : 0u);
          umma_commit_pair(bar_empty + 8 * s);
        }
        umma_commit_pair(bar_acc_full + 8 * as);
      }
      if (g + 1 < n_groups) umma_commit_pair(bar_qfree);   // arrives in both CTAs once this group's MMAs have completed
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue warps 2..5 (both CTAs): one row per thread
    const int quad = warp & 3;
    const size_t q_stride = (size_t)grid * p.capg;
    int tt = 0;
    for (int g = 0; g < n_groups; ++g) {
    unsigned long long* my_cand = p.cand + (size_t)g * p.group_cand_stride + (size_t)cta * p.capg;
    for (int t = 0; t < my_tiles; ++t, ++tt) {
      const int as = tt & 1;
      const int li = 2 * (pair + t * npairs) + (int)rank;
      const int tile = p.tile_first + li * p.tile_step;
      const int64_t row = (int64_t)tile * kTileRows + quad * 32 + lane;
      const bool live = li < p.num_tiles && row < p.n;
      const float invn = live ? __ldg(p.inv_norm + row) : 0.f;
      mbar_wait(bar_acc_full + 8 * as, ((uint32_t)tt >> 1) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // 32 columns per round (two x16 loads in flight, one wait); not unrolled: 128 live accumulator registers spill
#pragma unroll 1
      for (int c0 = 0; c0 < NQ; c0 += 32) {
        uint32_t v[16], w[16];
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * NQ + c0);
        TmemLd<16>::ld(taddr, v);
        TmemLd<16>::ld(taddr + 16u, w);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (p.thr_init == nullptr) {   // sampling pass: one key per (warp, query)
          sample_emit<16>(v, live, invn, my_cand, q_stride, c0, t * 4 + quad, lane);
          sample_emit<16>(w, live, invn, my_cand, q_stride, c0 + 16, t * 4 + quad, lane);
          continue;
        }
        if (live) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float score = __uint_as_float(j < 16 ? v[j] : w[j - 16]) * invn;
            if (score >= thr[c0 + j]) {
              const int pos = atomicAdd(&cnt[c0 + j], 1);
              if (pos < p.capg) my_cand[(size_t)(c0 + j) * q_stride + pos] = make_key32(score, (uint32_t)row);
            }
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa_u32(bar_acc_empty + 8 * as, 0));
    }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  for (int i = threadIdx.x; i < NQ * n_groups; i += blockDim.x) {
    const int g = i / NQ, qi = i - g * NQ;
    const int c = p.thr_init == nullptr ? my_tiles * 4 : cnt[qi];
    p.counts[(size_t)g * p.group_cnt_stride + (size_t)qi * grid + cta] = min(c, p.capg);
    if (c > p.capg && p.fallback) p.fallback[qi] = 1;
  }
  cluster_sync_all();   // no CTA leaves (or frees tensor memory) while its peer can still signal it
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(2 * NQ) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------ select kernel
struct SelectParams {
  const unsigned long long* cand;   // [nq][grid][capg]
  const int32_t* counts;            // [nq][grid]
  int32_t grid, capg;
  int32_t nq;                       // real queries in this block (padded operand rows get a +inf threshold)
  int32_t mode;                     // 0 = write the safe threshold (sampling pass), 1 = window + exact stage + emit
  float* thr_out;                   // [rows] (mode 0)
  const float* eps;                 // [nq] error bound of the approximate scores (0 = all-zero query)
  int32_t* fallback;                // [nq] (mode 1)
  const __half* rows;               // mode 1
  const float* q;                   // [nq][d_pad] the caller's fp32 queries
  int32_t d_pad, ch;
  int64_t id_base;
  int32_t k;
  int64_t* out_ids;
  double* out_scores;
  int32_t* out_counts;
};

// One CTA per query.  A lower bound of the k-th best approximate key among the survivors of all CTAs by an MSB-first
// RADIX SELECT (8-bit digits, shared-memory histogram; the pass loop stops as soon as the bucket holding the k-th key
// is small -- the undecided low bits are taken as zero, which only widens the window).
//   mode 0 (sampling pass): threshold = that score - 2 eps.
//   mode 1: gather every survivor inside the window below it, exact fp64 re-score of all of them, emit k.
// Survivors are staged in shared memory when they fit (the normal case: ~0.3 % of the corpus); otherwise every pass
// streams them from HBM/L2 -- slower, still exact.
__global__ void __launch_bounds__(kSelectThreads, 2) dense_select_kernel(const SelectParams p) {
  extern __shared__ __align__(16) uint8_t ssm[];
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ssm);  // [kSelStage] staged survivors
  unsigned long long* top = keys + kSelStage;                             // [kSelTop]   window members
  unsigned long long* ek = top + kSelTop;                                 // [kSelTop]   exact keys      (mode 1)
  uint32_t* ei = reinterpret_cast<uint32_t*>(ek + kSelTop);               // [kSelTop]   rows            (mode 1)
  __shared__ double qq_s;
  __shared__ int s_prefix[kSelectThreads + 1];
  __shared__ int s_hist[256];
  __shared__ int s_scal[4];
  __shared__ int s_ntop;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5, qi = blockIdx.x;
  const int K = p.k, G = p.grid;
  if (p.mode == 0 && qi >= p.nq) {   // padded operand row: nothing may survive
    if (tid == 0) p.thr_out[qi] = INFINITY;
    return;
  }
  if (p.mode == 1 && p.fallback[qi] != 0) return;   // a list overflowed: the brute-force kernel answers this query
  const int32_t* counts = p.counts + (size_t)qi * G;
  const unsigned long long* cand = p.cand + (size_t)qi * G * p.capg;
  // exclusive prefix of the per-CTA survivor counts (G <= blockDim): one element per thread
  {
    const int v = tid < G ? counts[tid] : 0;
    int x = v;
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) s_hist[warp] = x;
    if (tid == 0) s_ntop = 0;
    __syncthreads();
    if (warp == 0) {
      int w = lane < nw ? s_hist[lane] : 0;
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += y;
      }
      s_hist[32 + lane] = w;  // inclusive warp totals
    }
    __syncthreads();
    const int incl = x + (warp ? s_hist[32 + warp - 1] : 0);
    if (tid < G) s_prefix[tid] = incl - v;
    if (tid == G - 1) s_prefix[G] = incl;
    __syncthreads();
  }
  const int total = s_prefix[G];
  const bool staged = total <= kSelStage;
  if (staged) {
    for (int g = warp; g < G; g += nw) {
      const int c = s_prefix[g + 1] - s_prefix[g];
      const unsigned long long* src = cand + (size_t)g * p.capg;
      unsigned long long* dst = keys + s_prefix[g];
      for (int i = lane; i < c; i += 32) dst[i] = src[i];
    }
    __syncthreads();
  }
  // visit every survivor once: `body(key)`
#define SB_FOR_EACH_KEY(BODY)                                                       \
  if (staged) {                                                                     \
    for (int i_ = tid; i_ < total; i_ += nt) {                                      \
      const unsigned long long key = keys[i_];                                      \
      BODY                                                                          \
    }                                                                               \
  } else {                                                                          \
    for (int g_ = warp; g_ < G; g_ += nw) {                                         \
      const int c_ = s_prefix[g_ + 1] - s_prefix[g_];                               \
      const unsigned long long* src_ = cand + (size_t)g_ * p.capg;                  \
      for (int i_ = lane; i_ < c_; i_ += 32) {                                      \
        const unsigned long long key = src_[i_];                                    \
        BODY                                                                        \
      }                                                                             \
    }                                                                               \
  }

  unsigned long long prefix = 0ull, mask = 0ull;
  if (total > K) {
    int need = K;  // rank (from the top) of the key we are looking for inside the current bucket
    for (int shift = 56; shift >= 0; shift -= 8) {
      for (int i = tid; i < 256; i += nt) s_hist[i] = 0;
      __syncthreads();
      // warp-aggregated histogram update: in the leading passes nearly all keys share a digit, and per-key shared
      // atomics on one bin serialise; lanes with equal digits elect one lane to add their count
      SB_FOR_EACH_KEY(if ((key & mask) == prefix) {
        const int dgt = (int)((key >> shift) & 0xffull);
        const unsigned grp = __match_any_sync(__activemask(), dgt);
        if ((int)(threadIdx.x & 31) == __ffs(grp) - 1) atomicAdd(&s_hist[dgt], __popc(grp));
      })
      __syncthreads();
      if (warp == 0) warp_select_bin<true>(s_hist, need, lane, s_scal);
      __syncthreads();
      prefix |= (unsigned long long)s_scal[0] << shift;
      mask |= 0xffull << shift;
      need = s_scal[1];
      const int bucket = s_scal[2];
      __syncthreads();
      if (bucket <= 16) break;
    }
  }
  // `prefix` (undecided low bits zero) <= the k-th best key; total <= k: every survivor is a member (prefix = 0)
  const float eps = p.eps[qi];
  const unsigned long long lo_key = total > K ? window_lo_key(prefix, eps) : 0ull;
  if (p.mode == 0) {
    // fewer than k sampled rows: no threshold.  The score field of lo_key is (k-th best of the sample) - 2 eps.
    if (tid == 0) p.thr_out[qi] = total > K ? key32_score(lo_key) : -INFINITY;
    return;
  }
  SB_FOR_EACH_KEY(if (key >= lo_key) {
    const int at = atomicAdd(&s_ntop, 1);
    if (at < kSelTop) top[at] = key;
  })
#undef SB_FOR_EACH_KEY
  __syncthreads();
  const int ntop = s_ntop;
  if (ntop > kSelTop) {
    if (tid == 0) p.fallback[qi] = 1;
    return;
  }
  int P = 32;
  while (P < ntop) P <<= 1;
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
  // the staged survivors are dead (the window lives in `top`): their shared memory becomes the query staging area
  rescore_and_emit(top, ntop, P, ek, ei, &qq_s, reinterpret_cast<float*>(keys), ra);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int encode_map(CUtensorMap* map, const void* ptr, int64_t rows, int64_t cols, int box_rows) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* pfn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &pfn, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(pfn);
  }
  SB_REQUIRE(fn != nullptr, SB_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SB_REQUIRE(r == CUDA_SUCCESS, SB_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return SB_OK;
}

template <int QBN>
int launch_mma(const CUtensorMap& tm_rows, const CUtensorMap& tm_q, const MmaScanParams& mp, int grid, size_t smem,
               cudaStream_t st) {
  auto kern = dense_scan_mma_kernel<QBN>;
  SB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, kMmaThreads, smem, st>>>(tm_rows, tm_q, mp);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

int dispatch_mma(int qbn, const CUtensorMap& tm_rows, const CUtensorMap& tm_q, const MmaScanParams& mp, int grid,
                 size_t smem, cudaStream_t st) {
  switch (qbn) {
    case 16: return launch_mma<16>(tm_rows, tm_q, mp, grid, smem, st);
    case 32: return launch_mma<32>(tm_rows, tm_q, mp, grid, smem, st);
    case 64: return launch_mma<64>(tm_rows, tm_q, mp, grid, smem, st);
  }
  sb_set_error("dense_mma: unsupported query block %d", qbn);
  return SB_ERR_UNSUPPORTED;
}

// the pair kernel: 2-CTA clusters, grid = 2 x (co-resident clusters)
int launch_mma_pair(const CUtensorMap& tm_rows, const CUtensorMap& tm_q, const MmaScanParams& mp, int grid, size_t smem,
                    cudaStream_t st) {
  auto kern = dense_scan_mma2_kernel<128>;
  SB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, kMmaThreads, smem, st>>>(tm_rows, tm_q, mp);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

// co-resident 2-CTA clusters of the pair kernel at its largest shared-memory footprint (queried once per context)
int pair_clusters(sb_ctx* ctx, size_t smem) {
  if (ctx->max_clusters2 > 0) return ctx->max_clusters2;
  auto kern = dense_scan_mma2_kernel<128>;
  int n = 0;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(ctx->num_sms & ~1), 1, 1);
    cfg.blockDim = dim3(kMmaThreads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) n = 0;
  }
  (void)cudaGetLastError();
  if (n <= 0 || n > ctx->num_sms / 2) n = ctx->num_sms / 2;
  ctx->max_clusters2 = n;
  return n;
}

// TMA ring of a scan CTA whose query operand takes q_bytes of shared memory: as many 16 KB stages as fit, at least 3 and
// at most kMaxStages, plus 2 KB of barriers / thresholds / counts and 1 KB of alignment slack
struct Ring {
  int stages;
  size_t smem;
};
Ring ring_for(const sb_ctx* ctx, size_t q_bytes) {
  const int stages = std::max(3, std::min((int)((ctx->smem_optin - q_bytes - 3072) / kATileBytes), kMaxStages));
  return {stages, q_bytes + (size_t)stages * kATileBytes + 2048 + 1024};
}

}  // namespace

bool dense_mma_eligible(const sb_ctx* ctx, const DenseIndex& ix, int B) {
  if (B < 16) return false;
  if (ix.d_pad % kBK != 0 || ix.n_pad % kTileRows != 0) return false;
  if (ix.n < 64 * kTileRows) return false;  // tiny corpora: the CUDA-core scan is already launch bound
  const size_t need = (size_t)ix.d_pad * 16 * 2 + 3 * (size_t)kATileBytes + 4096;
  return need <= ctx->smem_optin;
}

int dense_mma_topk_enqueue(sb_ctx* ctx, DenseIndex& ix, const float* q_pad, int B, int k, int64_t* out_ids,
                           double* out_scores, int32_t* out_counts, cudaStream_t st) {
  const int kb_count = ix.d_pad / kBK;
  const int total_tiles = (int)(ix.n_pad / kTileRows);
  // largest single-CTA query block whose resident operand leaves >= 3 pipeline stages
  int qbn_max = 64;
  while (qbn_max > 16 && (size_t)qbn_max * ix.d_pad * 2 + 3 * (size_t)kATileBytes + 4096 > ctx->smem_optin) qbn_max >>= 1;
  // the pair kernel holds 64 operand rows per CTA: usable whenever the 64-row block fits
  const bool pair_ok = qbn_max == 64 && total_tiles >= 2;
  const int gsz = pair_ok ? 128 : qbn_max;          // operand rows per group
  const int grid1 = std::min(ctx->num_sms, total_tiles);
  int grid2 = 0;
  Ring ring2 = {0, 0};
  if (pair_ok) {
    ring2 = ring_for(ctx, (size_t)64 * ix.d_pad * 2);
    grid2 = 2 * std::min(pair_clusters(ctx, ring2.smem), (total_tiles + 1) / 2);
  }
  const int grid = std::max(grid1, grid2);          // list slots per query: both kernels index [row][grid][capg]
  const int grid_min = grid2 > 0 ? std::min(grid1, grid2) : grid1;
  // sampling pass geometry: a few tiles per CTA spread evenly over the corpus; every warp of a sampled tile reports the
  // best of its 32 rows, so a query gets n_s = 4 * sample_tiles keys -- aim for n_s >= 4 k
  const int per_cta = std::max(kSampleTilesPerCta, std::min(8, (k + grid - 1) / grid));
  const int sample_tiles = std::min(per_cta * grid, total_tiles);
  const int sample_step = total_tiles / sample_tiles;
  const int sgrid1 = std::min(grid1, sample_tiles);
  const int sgrid2 = pair_ok ? std::min(grid2, (sample_tiles + 1) & ~1) : 0;
  const int sgrid = std::max(sgrid1, sgrid2);
  const int sgrid_min = sgrid2 > 0 ? std::min(sgrid1, sgrid2) : sgrid1;
  // per-(CTA, query) list capacity.  Sampling pass: 4 keys per sampled tile of the CTA.  Full pass: the threshold is the
  // k-th best of n_s maxima of 32 rows, passed by a fraction p of the rows with (1 - p)^32 = 1 - k / n_s; 8x the expected
  // rows_per_cta * p plus slack.  An overflowing list raises the query's fallback flag, so the capacity only trades
  // memory against the odds of a brute-force answer; no threshold at all (k >= n_s) means every row survives.
  const int64_t worst = (int64_t)((total_tiles + grid_min - 1) / grid_min + 1) * kTileRows;
  const int64_t samp_keys = (int64_t)((sample_tiles + sgrid_min - 1) / sgrid_min + 1) * 4;
  const double f = (double)k / (4.0 * sample_tiles);
  const double pass = f >= 0.95 ? 1.0 : -log(1.0 - f) / 32.0;
  const int64_t expect = (int64_t)((double)worst * pass) + 1;
  const int capg = (int)std::min<int64_t>(worst, std::max<int64_t>(8 * expect + 256, samp_keys));
  int rc;
  SB_REQUIRE(grid <= kSelectThreads, SB_ERR_UNSUPPORTED, "dense_mma: %d CTAs exceed the select kernel's prefix width", grid);
  const int n_groups = (B + gsz - 1) / gsz;
  const size_t cand_per_group = (size_t)gsz * grid * capg * 8;
  int gmax = (int)std::max<size_t>(1, (size_t)(1024ull << 20) / cand_per_group);
  gmax = std::min(gmax, n_groups);
  // scratch: fp16 operand rows | thresholds + counts | survivors
  if ((rc = ctx->misc2_dev.reserve((size_t)n_groups * gsz * ix.d_pad * 2 + 256))) return rc;
  if ((rc = ctx->misc3_dev.reserve(((size_t)gsz * 4 + (size_t)gsz * grid * 4) * gmax + 256))) return rc;
  if ((rc = ctx->cand_dev.reserve(cand_per_group * gmax))) return rc;
  __half* q16 = ctx->misc2_dev.as<__half>();
  float* thr = ctx->misc3_dev.as<float>();
  int32_t* counts = reinterpret_cast<int32_t*>(thr + (size_t)gsz * gmax);
  unsigned long long* cand = ctx->cand_dev.as<unsigned long long>();
  if (ix.tm_rows_ptr != ix.rows) {  // (re)build the corpus tensor map once per loaded index
    if ((rc = encode_map(reinterpret_cast<CUtensorMap*>(ix.tm_rows), ix.rows, ix.n_pad, ix.d_pad, kTileRows))) return rc;
    ix.tm_rows_ptr = ix.rows;
  }
  const CUtensorMap& tm_rows = *reinterpret_cast<const CUtensorMap*>(ix.tm_rows);
  const size_t sel_smem = (size_t)kSelStage * 8 + (size_t)kSelTop * 20 + 64;
  SB_CUDA(cudaFuncSetAttribute(dense_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sel_smem));
  // normalised fp16 operand rows of the whole batch (rows beyond B are zero), eps, cleared fallback flags
  float* eps = nullptr;
  int32_t* fb = nullptr;
  if ((rc = dense_prep_queries(ctx, ix, q_pad, B, n_groups * gsz, /*mma=*/true, nullptr, q16, &eps, &fb, st))) return rc;

  for (int c0 = 0; c0 < B; c0 += gmax * gsz) {
    const int nq_chunk = std::min(B - c0, gmax * gsz);   // real queries of this chunk of groups
    const int ng = (nq_chunk + gsz - 1) / gsz;
    struct Group { int qbn, nq; bool pair; CUtensorMap tm_q; Ring ring; };
    std::vector<Group> gs((size_t)ng);
    int rows_total = 0;  // operand rows of the chunk (padding only at the very end)
    for (int g = 0; g < ng; ++g) {
      Group& G = gs[(size_t)g];
      const int left = nq_chunk - g * gsz;
      __half* q16g = q16 + (size_t)(c0 + g * gsz) * ix.d_pad;
      G.pair = pair_ok && left > 64;
      if (G.pair) {
        G.qbn = 128;
        G.nq = std::min(128, left);
        if ((rc = encode_map(&G.tm_q, q16g, 128, ix.d_pad, 64))) return rc;   // box = one CTA's 64 operand rows
        G.ring = ring2;
      } else {
        G.qbn = qbn_max;
        while (G.qbn > 16 && G.qbn / 2 >= left) G.qbn >>= 1;
        G.nq = std::min(G.qbn, left);
        if ((rc = encode_map(&G.tm_q, q16g, G.qbn, ix.d_pad, G.qbn))) return rc;
        G.ring = ring_for(ctx, (size_t)G.qbn * ix.d_pad * 2);
      }
      rows_total = g * gsz + G.qbn;
    }
    MmaScanParams mp;
    mp.inv_norm = ix.inv_norm;
    mp.n = ix.n;
    mp.kb_count = kb_count;
    mp.capg = capg;
    mp.n_groups = 1;
    mp.group_cand_stride = 0;
    mp.group_cnt_stride = 0;
    SelectParams sp;
    sp.cand = cand;
    sp.counts = counts;
    sp.capg = capg;
    sp.nq = nq_chunk;
    sp.thr_out = thr;
    sp.eps = eps + c0;
    sp.fallback = fb + c0;
    sp.rows = ix.rows;
    sp.q = q_pad + (size_t)c0 * ix.d_pad;
    sp.d_pad = ix.d_pad;
    sp.ch = ix.d_pad / 8;
    sp.id_base = ix.id_base;
    sp.k = k;
    sp.out_ids = out_ids + (size_t)c0 * k;
    sp.out_scores = out_scores + (size_t)c0 * k;
    sp.out_counts = out_counts + c0;
    // (1) sampling passes -> safe thresholds for every query of the chunk (one select launch).  Both kernels write
    // list slot `cta` of [row][launch grid][capg], so every group is launched with exactly sgrid CTAs (idle ones
    // report empty lists).
    mp.thr_init = nullptr;
    mp.fallback = nullptr;   // capg >= the sampled rows of a CTA: the sampling pass cannot overflow
    mp.num_tiles = sample_tiles;
    mp.tile_first = 0;
    mp.tile_step = sample_step;
    {
      ProfScope ps(ctx, SB_PROF_DENSE_SAMPLE, st, ng + 1);   // the sampling passes + their threshold select, as one span
      // the leading pair groups of the chunk share ONE sampling launch (a sampling launch is ~27 us of fixed cost: launch,
      // TMEM allocation, cluster syncs, the first operand load -- paid once instead of once per 128 queries)
      int n_pair = 0;
      while (n_pair < ng && gs[(size_t)n_pair].pair) ++n_pair;
      if (n_pair > 0) {
        CUtensorMap tm_q_all;
        if ((rc = encode_map(&tm_q_all, q16 + (size_t)c0 * ix.d_pad, (int64_t)n_pair * 128, ix.d_pad, 64))) return rc;
        mp.cand = cand;
        mp.counts = counts;
        mp.stages = ring2.stages;
        mp.n_groups = n_pair;
        mp.group_cand_stride = (int64_t)gsz * sgrid * capg;
        mp.group_cnt_stride = (int64_t)gsz * sgrid;
        if ((rc = launch_mma_pair(tm_rows, tm_q_all, mp, sgrid, ring2.smem, st))) return rc;
        mp.n_groups = 1;
      }
      // the single-CTA groups: all of them without the pair kernel, else only a trailing group of <= 64 queries
      for (int g = n_pair; g < ng; ++g) {
        const Group& G = gs[(size_t)g];
        mp.cand = cand + (size_t)g * gsz * sgrid * capg;
        mp.counts = counts + (size_t)g * gsz * sgrid;
        mp.stages = G.ring.stages;
        if ((rc = dispatch_mma(G.qbn, tm_rows, G.tm_q, mp, sgrid, G.ring.smem, st))) return rc;
      }
      sp.grid = sgrid;
      sp.mode = 0;
      dense_select_kernel<<<rows_total, kSelectThreads, sel_smem, st>>>(sp);
    }
    SB_CUDA(cudaGetLastError());
    // (2) the full passes, then one select + exact re-score launch for the chunk
    mp.num_tiles = total_tiles;
    mp.tile_first = 0;
    mp.tile_step = 1;
    for (int g = 0; g < ng; ++g) {
      const Group& G = gs[(size_t)g];
      mp.thr_init = thr + (size_t)g * gsz;
      mp.fallback = fb + c0 + (size_t)g * gsz;
      mp.cand = cand + (size_t)g * gsz * grid * capg;
      mp.counts = counts + (size_t)g * gsz * grid;
      mp.stages = G.ring.stages;
      ProfScope ps(ctx, SB_PROF_DENSE_SCAN, st);
      if (G.pair) rc = launch_mma_pair(tm_rows, G.tm_q, mp, grid, G.ring.smem, st);
      else rc = dispatch_mma(G.qbn, tm_rows, G.tm_q, mp, grid, G.ring.smem, st);
      if (rc) return rc;
    }
    sp.grid = grid;
    sp.mode = 1;
    {
      ProfScope ps(ctx, SB_PROF_DENSE_MERGE, st);
      dense_select_kernel<<<nq_chunk, kSelectThreads, sel_smem, st>>>(sp);
    }
    SB_CUDA(cudaGetLastError());
  }
  return dense_fallback_enqueue(ctx, ix, q_pad, B, k, fb, out_ids, out_scores, out_counts, st);
}
