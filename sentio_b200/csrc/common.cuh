// common.cuh -- shared host/device helpers for libsentio_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/sentio_b200.h"

// ------------------------------------------------------------------ error plumbing
void sb_set_error(const char* fmt, ...);

#define SB_CUDA(expr)                                                                         \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      sb_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__, __LINE__,    \
                   cudaGetErrorString(_e));                                                   \
      return SB_ERR_CUDA;                                                                     \
    }                                                                                         \
  } while (0)

#define SB_REQUIRE(cond, code, ...)  \
  do {                               \
    if (!(cond)) {                   \
      sb_set_error(__VA_ARGS__);     \
      return (code);                 \
    }                                \
  } while (0)

// ------------------------------------------------------------------ device buffers (grow-only scratch)
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes) {
    if (bytes <= cap) return SB_OK;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + (bytes >> 2) + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      sb_set_error("cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
      return SB_ERR_CUDA;
    }
    cap = want;
    return SB_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

struct PinBuf {
  void* p = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes) {
    if (bytes <= cap) return SB_OK;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + (bytes >> 2) + 256;
    cudaError_t e = cudaMallocHost(&p, want);
    if (e != cudaSuccess) {
      sb_set_error("cudaMallocHost(%zu) failed: %s", want, cudaGetErrorString(e));
      return SB_ERR_CUDA;
    }
    cap = want;
    return SB_OK;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

// ------------------------------------------------------------------ index state
struct DenseIndex {
  int64_t n = 0;        // valid rows
  int64_t n_pad = 0;    // rows allocated (multiple of 32, zero filled)
  int32_t d = 0;        // logical dimension
  int32_t d_pad = 0;    // stored row length in halves (multiple of 8 -> 16 B aligned rows)
  int64_t id_base = 0;
  __half* rows = nullptr;    // [n_pad][d_pad]
  float* inv_norm = nullptr; // [n_pad], 1/||row|| of the STORED fp16 row (0 for zero rows)
  // cached CUtensorMap (128 bytes, 64-byte aligned) over rows[] for the tcgen05 batched scan; valid iff tm_rows_ptr == rows
  alignas(64) unsigned char tm_rows[128] = {0};
  const void* tm_rows_ptr = nullptr;
};

struct Bm25Index {
  int64_t n_docs = 0, n_terms = 0, nnz = 0;
  int64_t id_base = 0;
  int32_t variant = 0;
  double k1 = 1.5, b = 0.75, delta = 1.0, avgdl = 0.0;
  int64_t* indptr = nullptr;   // [V+1]
  int32_t* post_doc = nullptr; // [nnz]
  double* post_ratio = nullptr; // [nnz] query-independent tf*(k1+1)/(tf+dnorm[doc]) (fp64, exact op order)
  double* dnorm = nullptr;     // [n_docs]  k1*(1-b+b*dl/avgdl), same op order as rank_bm25
  double* idf = nullptr;       // [V]
  // head terms (df >= n_docs / 4) additionally keep a DENSE ratio row: dense_ratio[slot][doc] (0.0 where the doc has no
  // posting); dense_of_term[t] = slot or -1.  The scoring kernel streams these rows with fully predictable addresses
  int32_t n_dense = 0;
  int32_t* dense_of_term = nullptr;  // [V]
  double* dense_ratio = nullptr;     // [n_dense][n_docs]
};

struct CeModel;      // cross_encoder.cu
struct CeDocTokens;  // cross_encoder.cu
struct Bm25Build;    // bm25_build.cu

struct sb_ctx {
  int device = 0;
  int num_sms = 0;
  size_t smem_optin = 0;
  cudaStream_t stream = nullptr;
  std::mutex mu;
  DenseIndex dense[SB_MAX_DENSE_SLOTS];
  Bm25Index bm25;
  CeModel* ce = nullptr;   // reranker (sb_ce_load)
  CeModel* enc = nullptr;  // query / document embedder (sb_enc_load)
  CeDocTokens* ce_tokens = nullptr;
  Bm25Build* bm25_build = nullptr;  // GPU index build in progress (sb_bm25_build_tokens .. sb_bm25_build_finish)
  int dense_mode = 0;  // 0 = auto, 1 = CUDA-core scan only
  int max_clusters2 = 0;  // co-resident 2-CTA clusters of the pair kernel (0 = not queried yet)
  // bookkeeping: kernels launched by this library, optional per-kernel CUDA-event timing (bench.py roofline leg)
  uint64_t launches = 0;
  bool prof_on = false;
  struct ProfRec { int id; cudaEvent_t a, b; };
  std::vector<ProfRec> prof_recs;
  std::vector<cudaEvent_t> prof_pool;
  // scratch
  DevBuf q_dev, cand_dev, out_ids_dev, out_sc_dev, out_cnt_dev, misc_dev, misc2_dev, misc3_dev, acc_dev;
  DevBuf qn_dev;     // dense: normalised fp32 queries [B][d_pad] fed to the scans
  DevBuf qaux_dev;   // dense: per-query eps [B] fp32 | fallback flags [B] i32
  DevBuf doc_chars_dev;  // K7: characters of every document's usable text (0 = blank), sb_doc_chars_load
  int64_t doc_chars_n = 0, doc_chars_base = 0;
  PinBuf pin_in, pin_out;
  // sb_hybrid_topk: staging of one whole-path call (its own buffers and lock: the inner entry points take `mu`)
  std::mutex hyb_mu;
  PinBuf hyb_pin;
  DevBuf hyb_dev;
};

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    cudaGetDevice(&cur);
    if (prev >= 0 && cur != prev) cudaSetDevice(prev);
  }
};

// kernel ids for sb_profile_read
enum { SB_PROF_DENSE_SCAN = 0, SB_PROF_DENSE_MERGE = 1, SB_PROF_BM25_SCORE = 2, SB_PROF_BM25_SELECT = 3,
       SB_PROF_FUSE = 4, SB_PROF_CE = 5, SB_PROF_DENSE_SAMPLE = 6, SB_PROF_COUNT = 7 };

static inline cudaEvent_t prof_event(sb_ctx* ctx) {
  if (!ctx->prof_pool.empty()) {
    cudaEvent_t e = ctx->prof_pool.back();
    ctx->prof_pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}
// bracket `n_kernels` launches of kernel `id` on stream st with an event pair when profiling is enabled
struct ProfScope {
  sb_ctx* ctx;
  cudaStream_t st;
  cudaEvent_t b = nullptr;
  ProfScope(sb_ctx* c, int id, cudaStream_t s, int n_kernels = 1) : ctx(c), st(s) {
    ctx->launches += (uint64_t)n_kernels;
    if (ctx->prof_on) {
      cudaEvent_t a = prof_event(ctx);
      b = prof_event(ctx);
      cudaEventRecord(a, st);
      ctx->prof_recs.push_back({id, a, b});
    }
  }
  ~ProfScope() {
    if (b) cudaEventRecord(b, st);
  }
};

// true when [p, p + bytes) is page-locked host memory the copy engines can reach directly (cudaMallocHost / registered)
static inline bool host_ptr_is_pinned(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    (void)cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeHost;
}

static inline cudaStream_t pick_stream(sb_ctx* ctx, void* stream) {
  return stream ? reinterpret_cast<cudaStream_t>(stream) : ctx->stream;
}

// ------------------------------------------------------------------ device helpers
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t f32_orderable(float f) {
  uint32_t u = __float_as_uint(f);
  return u ^ ((u >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float orderable_f32(uint32_t u) {
  u ^= (u >> 31) ? 0x80000000u : 0xffffffffu;
  return __uint_as_float(u);
}
__device__ __forceinline__ uint64_t f64_orderable(double d) {
  uint64_t u = (uint64_t)__double_as_longlong(d);
  return u ^ ((u >> 63) ? 0xffffffffffffffffull : 0x8000000000000000ull);
}
__device__ __forceinline__ double orderable_f64(uint64_t u) {
  u ^= (u >> 63) ? 0x8000000000000000ull : 0xffffffffffffffffull;
  return __longlong_as_double((long long)u);
}
// composite key: larger = better.  hi 32 = orderable score, lo 32 = ~idx (lower idx wins ties).
__device__ __forceinline__ uint64_t make_key32(float score, uint32_t idx) {
  return ((uint64_t)f32_orderable(score) << 32) | (uint64_t)(~idx);
}
__device__ __forceinline__ uint32_t key32_idx(uint64_t k) { return ~(uint32_t)(k & 0xffffffffu); }
__device__ __forceinline__ float key32_score(uint64_t k) { return orderable_f32((uint32_t)(k >> 32)); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}


// Radix-select helper, called by ONE full warp: scan the 256-bin histogram from the top (DESC) or the bottom and find the
// bin where the running count first reaches `need`.  out[0] = bin, out[1] = rank inside the bin (need - count of the bins
// before it), out[2] = the bin's count.  Lane l owns 8 consecutive bins in scan order; one shuffle scan across lanes.
template <bool DESC>
__device__ __forceinline__ void warp_select_bin(const int* hist, int need, int lane, int* out) {
  int c[8];
  int s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int b = DESC ? 255 - 8 * lane - i : 8 * lane + i;
    c[i] = hist[b];
    s += c[i];
  }
  int incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  const int excl = incl - s;
  const bool mine = excl < need && need <= incl;
  const unsigned m = __ballot_sync(0xffffffffu, mine);
  if (mine) {
    int cum = excl;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (cum + c[i] >= need) {
        out[0] = DESC ? 255 - 8 * lane - i : 8 * lane + i;
        out[1] = need - cum;
        out[2] = c[i];
        break;
      }
      cum += c[i];
    }
  }
  if (m == 0u && lane == 31) {  // fewer than `need` keys in total (callers avoid it): same answer as a full serial scan
    out[0] = DESC ? 0 : 255;
    out[1] = need - incl;
    out[2] = hist[DESC ? 0 : 255];
  }
}

// ---- mbarrier / bulk-copy (TMA engine, SASS UBLKCP) wrappers
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
// 1-D bulk async copy global -> shared, completion signalled on an mbarrier (bytes % 16 == 0, 16 B aligned).
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar), "l"(policy)
      : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// barrier + OR reduction of a predicate over the participating threads
__device__ __forceinline__ bool named_bar_or(int id, int nthreads, bool pred) {
  uint32_t r;
  asm volatile(
      "{\n"
      ".reg .pred p, q;\n"
      "setp.ne.u32 p, %3, 0;\n"
      "bar.red.or.pred q, %1, %2, p;\n"
      "selp.u32 %0, 1, 0, q;\n"
      "}\n"
      : "=r"(r)
      : "r"(id), "r"(nthreads), "r"((uint32_t)pred)
      : "memory");
  return r != 0;
}

#endif  // __CUDACC__
