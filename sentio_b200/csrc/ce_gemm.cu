// ce_gemm.cu -- tcgen05 / TMEM / TMA GEMM for the cross-encoder (K5):  D[M,N] = A[M,K] * W[N,K]^T  (+ epilogue)
//
// A (activations) and W (nn.Linear weights) are both K-major fp16, accumulation is fp32 in tensor memory.
// One 128 x 128 output tile per CTA, K consumed in 64-element (128-byte, SWIZZLE_128B) chunks through a 3-stage
// TMA -> mbarrier -> tcgen05.mma ring; warp roles: warp 0 = TMA producer (one elected lane), warp 1 = TMEM allocator +
// MMA issuer (one elected lane), warps 2..5 = epilogue (tcgen05.ld 32x32b, one accumulator row per thread).
// Two CTAs are resident per SM (96 KB smem, 128 TMEM columns each) so one tile's epilogue overlaps another's mainloop.
//
// Epilogues:  BIAS_F16        out16 = acc + bias                      (QKV projection)
//             BIAS_GELU_F16   out16 = gelu_erf(acc + bias)            (FFN up-projection)
//             BIAS_RES_F32    out32 = acc + bias + residual32         (attention output / FFN down-projection, pre-LN)
//             BIAS_RES16_F16  out16 = fp16(acc + bias + residual16)   (the same two GEMMs on the fp16 residual stream:
//                             half the epilogue bytes; the pre-LN sum is rounded to fp16 once)
//
// Bound: tensor pipe (2*M*N*K flops); see DESIGN.md for the per-pair flop count.
#include <cuda.h>
#include <stdlib.h>

#include <algorithm>

#include "ce_gemm.cuh"

namespace {

constexpr int BM = 128, BN = 128, BK = 64;
constexpr int kStages = 3;
constexpr int kGemmThreads = 192;
constexpr uint32_t kTileABytes = BM * BK * 2, kTileBBytes = BN * BK * 2;
constexpr uint32_t kStageBytes = kTileABytes + kTileBBytes;
constexpr uint32_t kTmemCols = 128;
constexpr size_t kGemmSmem = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
      "l"(map), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (cf. cute::UMMA::SmemDescriptor): start address >> 4,
// LBO = 1 (unused for swizzled K-major), SBO = 1024 B (8 rows x 128 B swizzle atom) >> 4, version = 1, layout = 2.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3fff);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// kind::f16 instruction descriptor: D = f32, A = B = f16, both K-major, N >> 3 at [17,23), M >> 4 at [24,29).
__device__ __forceinline__ uint32_t make_idesc() {
  uint32_t d = 0;
  d |= 1u << 4;                     // c_format = F32
  d |= 0u << 7;                     // a_format = F16
  d |= 0u << 10;                    // b_format = F16
  d |= (uint32_t)(BN >> 3) << 17;   // n_dim
  d |= (uint32_t)(BM >> 4) << 24;   // m_dim
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

// erf-GELU (the HuggingFace "gelu") = 0.5 x (1 + erf(x / sqrt 2)), evaluated on a PAIR of outputs in packed half precision
// with ONE transcendental:  erf(x / sqrt 2) ~ tanh(x (c0 + c1 x^2 + c2 x^4)),  c fitted by least squares on the GELU itself
// over |x| <= 5.5 (scripts/fit_gelu.py): max |error| 3.0e-5 in exact arithmetic -- 16 x below the stock "tanh GELU"
// (4.7e-4) and below half an fp16 ulp of the result wherever |gelu| > 0.06.  8 packed instructions per pair
// (HMUL2 HMNMX2 2 x HFMA2 HMUL2 MUFU.TANH HMUL2 HFMA2); x^2 is clamped at 36 where tanh has saturated in fp16.
// History: fp32 libdevice erff made the FFN-up epilogue issue bound (r01 run 21: 78 % issue utilisation, tensor pipe
// 28 %); the Abramowitz-Stegun 7.1.26 form in half2 (reciprocal + exponential + 5-term Horner, 17 instructions per pair)
// was the round-1 fix; this form cut FFN-up from 340 to 269 us (ncu launch lists of r02 run 12, same box) and the rerank
// workload from 2741 to 2865 queries/s.  Error study (scripts/fit_gelu.py, every operation rounded to fp16, tanh with the
// 2^-11 relative error of tanh.approx): rms |error| 2.0e-4 on N(0,1) inputs vs 2.6e-4 for the A-S form and 1.3e-4 for the
// exact function rounded to fp16 -- the storage rounding dominates either way (tolerance of the path: 1e-3 on the score).
__device__ __forceinline__ __half2 gelu_erf_h2(__half2 x) {
  const __half2 x2 = __hmin2(__hmul2(x, x), __float2half2_rn(36.0f));
  __half2 q = __hfma2(__float2half2_rn(-0.00035873236644f), x2, __float2half2_rn(0.0370503451315f));
  q = __hfma2(q, x2, __float2half2_rn(0.79745847075f));
  const __half2 u = __hmul2(x, q);
  uint32_t tb;
  const uint32_t ub = *reinterpret_cast<const uint32_t*>(&u);
  asm("tanh.approx.f16x2 %0, %1;" : "=r"(tb) : "r"(ub));
  const __half2 th = *reinterpret_cast<const __half2*>(&tb);
  const __half2 hx = __hmul2(__float2half2_rn(0.5f), x);
  return __hfma2(hx, th, hx);
}
// bias-added fp32 pair -> fp16 pair, through the activation of the epilogue
template <int EPI>
__device__ __forceinline__ __half2 act_pack(float a, float b) {
  const __half2 h = __floats2half2_rn(a, b);
  return EPI == CE_EPI_BIAS_GELU_F16 ? gelu_erf_h2(h) : h;
}

template <int EPI>
__global__ void __launch_bounds__(kGemmThreads, 2)
ce_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w, int M_cap, int N, int K,
               const float* __restrict__ bias, const float* __restrict__ residual, __half* __restrict__ out16,
               float* __restrict__ out32, const int* __restrict__ m_dev) {
  const int M = m_dev ? min(M_cap, __ldg(m_dev)) : M_cap;
  extern __shared__ uint8_t gsm_raw[];
  // SWIZZLE_128B tiles need 1024-byte alignment
  const uint32_t raw = smem_u32(gsm_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* gsm = gsm_raw + (base - raw);
  uint64_t* bars = reinterpret_cast<uint64_t*>(gsm + kStages * kStageBytes);
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + kStages), bar_acc = smem_u32(bars + 2 * kStages);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int num_k = K / BK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_acc, 1);
    mbar_fence_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_acc = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < num_k; ++kb) {
        const int s = kb % kStages;
        const uint32_t use = (uint32_t)(kb / kStages);
        if (kb >= kStages) mbar_wait(bar_empty + 8 * s, (use & 1u) ^ 1u);
        const uint32_t sa = base + (uint32_t)s * kStageBytes, sb = sa + kTileABytes;
        mbar_expect_tx(bar_full + 8 * s, kStageBytes);
        tma_load_2d(sa, &map_a, kb * BK, m0, bar_full + 8 * s);
        tma_load_2d(sb, &map_w, kb * BK, n0, bar_full + 8 * s);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc();
      for (int kb = 0; kb < num_k; ++kb) {
        const int s = kb % kStages;
        const uint32_t use = (uint32_t)(kb / kStages);
        mbar_wait(bar_full + 8 * s, use & 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sa = base + (uint32_t)s * kStageBytes, sb = sa + kTileABytes;
        const uint64_t da = make_smem_desc(sa), db = make_smem_desc(sb);
#pragma unroll
        for (int k = 0; k < BK / 16; ++k) {
          // advance 16 fp16 = 32 bytes along K inside the 128-byte swizzle atom: +2 in the (addr >> 4) field
          umma_f16(tmem_acc, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) ? 1u : 0u);
        }
        umma_commit(bar_empty + 8 * s);  // frees this smem stage once the MMAs above have read it
      }
      umma_commit(bar_acc);  // accumulator complete
    }
  } else {
    // ---------------------------------------------------------------- epilogue warps 2..5
    const int quad = warp & 3;  // TMEM lane quadrant this warp may read
    mbar_wait(bar_acc, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int row = m0 + quad * 32 + lane;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t v[32];
      const uint32_t taddr = tmem_acc + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0;
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
          "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
          : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
            "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
            "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
            "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
          : "r"(taddr)
          : "memory");
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      if (row < M) {
        const int col = n0 + c0;
        if (EPI == CE_EPI_BIAS_RES_F32) {
          float* o = out32 + (size_t)row * N + col;
          const float* r = residual + (size_t)row * N + col;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 rb = *reinterpret_cast<const float4*>(r + j);
            const float4 bb = *reinterpret_cast<const float4*>(bias + col + j);
            float4 w;
            w.x = __uint_as_float(v[j + 0]) + bb.x + rb.x;
            w.y = __uint_as_float(v[j + 1]) + bb.y + rb.y;
            w.z = __uint_as_float(v[j + 2]) + bb.z + rb.z;
            w.w = __uint_as_float(v[j + 3]) + bb.w + rb.w;
            *reinterpret_cast<float4*>(o + j) = w;
          }
        } else if (EPI == CE_EPI_BIAS_RES16_F16) {
          __half* o = out16 + (size_t)row * N + col;
          const __half* r = reinterpret_cast<const __half*>(residual) + (size_t)row * N + col;
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            const uint4 rraw = *reinterpret_cast<const uint4*>(r + j);
            const __half2* rh = reinterpret_cast<const __half2*>(&rraw);
            uint4 pk;
            uint32_t* pw = reinterpret_cast<uint32_t*>(&pk);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 rf = __half22float2(rh[e]);
              const __half2 h = __floats2half2_rn(__uint_as_float(v[j + 2 * e]) + __ldg(bias + col + j + 2 * e) + rf.x,
                                                  __uint_as_float(v[j + 2 * e + 1]) + __ldg(bias + col + j + 2 * e + 1) + rf.y);
              pw[e] = *reinterpret_cast<const uint32_t*>(&h);
            }
            *reinterpret_cast<uint4*>(o + j) = pk;
          }
        } else {
          __half* o = out16 + (size_t)row * N + col;
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            float f[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              f[e] = __uint_as_float(v[j + e]) + __ldg(bias + col + j + e);
            }
            uint4 pk;
            __half2 h0 = act_pack<EPI>(f[0], f[1]), h1 = act_pack<EPI>(f[2], f[3]);
            __half2 h2 = act_pack<EPI>(f[4], f[5]), h3 = act_pack<EPI>(f[6], f[7]);
            pk.x = *reinterpret_cast<uint32_t*>(&h0);
            pk.y = *reinterpret_cast<uint32_t*>(&h1);
            pk.z = *reinterpret_cast<uint32_t*>(&h2);
            pk.w = *reinterpret_cast<uint32_t*>(&h3);
            *reinterpret_cast<uint4*>(o + j) = pk;
          }
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "n"(kTmemCols) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------ weight-stationary
// Persistent variant for K <= 384 (QKV / attention-out / FFN-up): the 128 x K weight tile of this CTA's n-tile stays in
// shared memory for the whole kernel and only activation tiles stream through the TMA ring, which halves the L2 -> SM
// traffic per output tile (the 128 x 128 x 384 tiles of the plain kernel are L2-bandwidth bound at ~64 flop/B); the
// accumulator is double buffered in tensor memory so the epilogue of tile i overlaps the MMAs of tile i + 1.
constexpr int kWsStages = 5;
constexpr int kWsAcc = 2;   // accumulator stages in tensor memory.  4 (all 512 columns, the MMA issuer up to three tiles ahead
                            // of the epilogue) was measured twice and changes nothing: QKV 196.6 -> 195.1 us, FFN-up 269.3 ->
                            // 268.0 (profiles/r02_run15_launches_rerank_{base,acc4}.csv) -- the K = 384 GEMMs wait for the
                            // epilogue of the CURRENT tile, not for accumulator space
constexpr int kWsEpiWarps = 16;                     // 4 per TMEM lane quadrant, 32 accumulator columns each
constexpr int kWsThreads = 64 + 32 * kWsEpiWarps;   // TMA warp + MMA warp + epilogue warps
constexpr uint32_t kStageRow = 80;                  // bytes per staged row (64 B of payload + 16 B pad: conflict-free 128-bit stores)
constexpr uint32_t kStageWarpBytes = 32 * kStageRow; // one epilogue warp's staging tile (32 rows)

template <int EPI>
__device__ __forceinline__ void epilogue_store_32(const uint32_t (&v)[32], int row, int col, int N,
                                                  const float* __restrict__ bias, const float* __restrict__ residual,
                                                  __half* __restrict__ out16, float* __restrict__ out32) {
  if (EPI == CE_EPI_BIAS_RES16_F16) {
    __half* o = out16 + (size_t)row * N + col;
    const __half* r = reinterpret_cast<const __half*>(residual) + (size_t)row * N + col;
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      const uint4 rraw = *reinterpret_cast<const uint4*>(r + j);
      const __half2* rh = reinterpret_cast<const __half2*>(&rraw);
      uint4 pk;
      uint32_t* pw = reinterpret_cast<uint32_t*>(&pk);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 rf = __half22float2(rh[e]);
        const __half2 h = __floats2half2_rn(__uint_as_float(v[j + 2 * e]) + __ldg(bias + col + j + 2 * e) + rf.x,
                                            __uint_as_float(v[j + 2 * e + 1]) + __ldg(bias + col + j + 2 * e + 1) + rf.y);
        pw[e] = *reinterpret_cast<const uint32_t*>(&h);
      }
      *reinterpret_cast<uint4*>(o + j) = pk;
    }
  } else if (EPI == CE_EPI_BIAS_RES_F32) {
    float* o = out32 + (size_t)row * N + col;
    const float* r = residual + (size_t)row * N + col;
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 rb = *reinterpret_cast<const float4*>(r + j);
      const float4 bb = *reinterpret_cast<const float4*>(bias + col + j);
      float4 w;
      w.x = __uint_as_float(v[j + 0]) + bb.x + rb.x;
      w.y = __uint_as_float(v[j + 1]) + bb.y + rb.y;
      w.z = __uint_as_float(v[j + 2]) + bb.z + rb.z;
      w.w = __uint_as_float(v[j + 3]) + bb.w + rb.w;
      *reinterpret_cast<float4*>(o + j) = w;
    }
  } else {
    __half* o = out16 + (size_t)row * N + col;
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      float f[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        f[e] = __uint_as_float(v[j + e]) + __ldg(bias + col + j + e);
      }
      uint4 pk;
      const __half2 h0 = act_pack<EPI>(f[0], f[1]), h1 = act_pack<EPI>(f[2], f[3]);
      const __half2 h2 = act_pack<EPI>(f[4], f[5]), h3 = act_pack<EPI>(f[6], f[7]);
      pk.x = *reinterpret_cast<const uint32_t*>(&h0);
      pk.y = *reinterpret_cast<const uint32_t*>(&h1);
      pk.z = *reinterpret_cast<const uint32_t*>(&h2);
      pk.w = *reinterpret_cast<const uint32_t*>(&h3);
      *reinterpret_cast<uint4*>(o + j) = pk;
    }
  }
}

template <int EPI, bool RESIDENT>
__global__ void __launch_bounds__(kWsThreads, 1)
ce_gemm_ws_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w, int M_cap, int N,
                  int K, const float* __restrict__ bias, const float* __restrict__ residual, __half* __restrict__ out16,
                  float* __restrict__ out32, const int* __restrict__ m_dev) {
  const int M = m_dev ? min(M_cap, __ldg(m_dev)) : M_cap;
  extern __shared__ uint8_t wsm_raw[];
  const uint32_t raw = smem_u32(wsm_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* sm = wsm_raw + (base - raw);
  const int num_k = K / BK;
  // RESIDENT: [W: num_k x 16 KB][A ring: stages x 16 KB]      streaming: [ring: stages x (A 16 KB + W 16 KB)]
  constexpr uint32_t kRingStage = RESIDENT ? kTileABytes : kStageBytes;
  const uint32_t w_bytes = RESIDENT ? (uint32_t)num_k * kTileBBytes : 0u;
  const uint32_t a0 = base + w_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + w_bytes + kWsStages * kRingStage);
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + kWsStages), bar_w = smem_u32(bars + 2 * kWsStages);
  const uint32_t bar_acc_full = smem_u32(bars + 2 * kWsStages + 1), bar_acc_empty = smem_u32(bars + 2 * kWsStages + 1 + kWsAcc);
  // (slot index chosen so that the epilogue staging area behind it, tmem_slot + 2 words, is 16-byte aligned)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kWsStages + 3 + 2 * kWsAcc);
  static_assert(((2 * kWsStages + 3 + 2 * kWsAcc) * 8 + 8) % 16 == 0 && (2 * kWsStages + 3 + 2 * kWsAcc) * 8 + 8 <= 256,
                "barrier block layout");
  uint8_t* stage_s = reinterpret_cast<uint8_t*>(tmem_slot + 2);                   // [kWsEpiWarps][32 rows][80 B]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = N / BN, m_tiles = (M + BM - 1) / BM;
  // RESIDENT: this CTA owns one n-tile for its lifetime and a strided share of the m-tiles.
  // streaming: tiles are enumerated n-fastest (consecutive CTAs share the same activation rows in L2).
  const int n_tile_fixed = blockIdx.x % n_tiles;
  const int peer = blockIdx.x / n_tiles;                                        // index among the CTAs of this n-tile
  const int peers = ((int)gridDim.x - n_tile_fixed + n_tiles - 1) / n_tiles;    // CTAs that own this n-tile
  const int total_tiles = n_tiles * m_tiles;
  const int my_tiles = RESIDENT ? (peer < m_tiles ? (m_tiles - 1 - peer) / peers + 1 : 0)
                                : ((int)blockIdx.x < total_tiles ? (total_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0);
  auto tile_m0 = [&](int t) -> int {
    return RESIDENT ? (peer + t * peers) * BM : (((int)blockIdx.x + t * (int)gridDim.x) / n_tiles) * BM;
  };
  auto tile_n0 = [&](int t) -> int {
    return RESIDENT ? n_tile_fixed * BN : (((int)blockIdx.x + t * (int)gridDim.x) % n_tiles) * BN;
  };

  if (threadIdx.x == 0) {
    for (int s = 0; s < kWsStages; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_w, 1);
    for (int s = 0; s < kWsAcc; ++s) {
      mbar_init(bar_acc_full + 8 * s, 1);
      mbar_init(bar_acc_empty + 8 * s, kWsEpiWarps);
    }
    mbar_fence_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(kWsAcc * BN)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      if (RESIDENT) {
        mbar_expect_tx(bar_w, w_bytes);
        for (int kb = 0; kb < num_k; ++kb)
          tma_load_2d(base + (uint32_t)kb * kTileBBytes, &map_w, kb * BK, n_tile_fixed * BN, bar_w);
      }
      int it = 0;
      for (int t = 0; t < my_tiles; ++t) {
        const int m0 = tile_m0(t), n0 = tile_n0(t);
        for (int kb = 0; kb < num_k; ++kb, ++it) {
          const int s = it % kWsStages;
          const uint32_t use = (uint32_t)(it / kWsStages);
          if (it >= kWsStages) mbar_wait(bar_empty + 8 * s, (use & 1u) ^ 1u);
          mbar_expect_tx(bar_full + 8 * s, kRingStage);
          tma_load_2d(a0 + (uint32_t)s * kRingStage, &map_a, kb * BK, m0, bar_full + 8 * s);
          if (!RESIDENT) tma_load_2d(a0 + (uint32_t)s * kRingStage + kTileABytes, &map_w, kb * BK, n0, bar_full + 8 * s);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc();
      if (RESIDENT) mbar_wait(bar_w, 0);
      int it = 0;
      for (int t = 0; t < my_tiles; ++t) {
        const int as = t % kWsAcc;
        if (t >= kWsAcc) mbar_wait(bar_acc_empty + 8 * as, (((uint32_t)(t / kWsAcc)) & 1u) ^ 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
        for (int kb = 0; kb < num_k; ++kb, ++it) {
          const int s = it % kWsStages;
          const uint32_t use = (uint32_t)(it / kWsStages);
          mbar_wait(bar_full + 8 * s, use & 1u);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint64_t da = make_smem_desc(a0 + (uint32_t)s * kRingStage);
          const uint64_t db = make_smem_desc(RESIDENT ? base + (uint32_t)kb * kTileBBytes
                                                       : a0 + (uint32_t)s * kRingStage + kTileABytes);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            umma_f16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (kb | k) ? 1u : 0u);
          umma_commit(bar_empty + 8 * s);
        }
        umma_commit(bar_acc_full + 8 * as);
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue: 16 warps; warp e reads TMEM lane quadrant
    // (warp & 3), accumulator columns [32 * (e >> 2), +32).  Phase 1: thread = accumulator row, bias (+GELU) applied,
    // 64 bytes of the row parked in a padded shared-memory tile.  Phase 2: the tile is drained two rows per instruction
    // so that every global access is a full, coalesced 64-byte row segment (thread-per-row stores straight to global are
    // LSU / latency bound; see profiles/r01_run5_ce_gemm_ncu.md vs r01_run8_ce_gemm_ws_ncu.md).
    const int e = warp - 2, quad = warp & 3, colgrp = e >> 2;
    uint8_t* st = stage_s + (size_t)e * kStageWarpBytes;
    const int sub = lane >> 4, c16 = lane & 15;
    float bias_lane = 0.f;  // bias of column (col0 + lane); broadcast with shuffles in phase 1
    int bias_col0 = -1;
    // weight-stationary bias / GELU kernels: the warp's column group is fixed for the whole kernel -> its 32 bias values
    // live in registers instead of being broadcast with 32 shuffles per tile (QKV 196.6 -> 185.6 us, FFN-up 269.3 -> 257.9,
    // profiles/r02_run15_launches_rerank_{base,acc4b}.csv).  The residual epilogues keep the shuffles (an earlier attempt
    // with registers there doubled the out-projection's time, profiles/r02_run9_launches_rerank_4acc_biasregs.csv).
    constexpr bool kBiasRegs = RESIDENT && (EPI == CE_EPI_BIAS_F16 || EPI == CE_EPI_BIAS_GELU_F16);
    float bias_r[kBiasRegs ? 32 : 1];
    if (kBiasRegs) {
#pragma unroll
      for (int j = 0; j < (kBiasRegs ? 32 : 0); j += 4) {
        const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + n_tile_fixed * BN + colgrp * 32 + j));
        bias_r[j] = b4.x; bias_r[j + 1] = b4.y; bias_r[j + 2] = b4.z; bias_r[j + 3] = b4.w;
      }
    }
    for (int t = 0; t < my_tiles; ++t) {
      const int as = t % kWsAcc;
      const int row0 = tile_m0(t) + quad * 32;
      const int col0 = tile_n0(t) + colgrp * 32;
      if (col0 != bias_col0) {
        bias_lane = __ldg(bias + col0 + lane);
        bias_col0 = col0;
      }
      // BIAS_RES16: this thread's residual row segment (32 fp16 = 64 bytes of row row0 + lane) is requested before the
      // accumulator wait, so its latency hides behind the MMAs of the tile
      uint4 rres[EPI == CE_EPI_BIAS_RES16_F16 ? 4 : 1];
      if (EPI == CE_EPI_BIAS_RES16_F16) {
        const int row = row0 + lane;
        const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(residual) + (size_t)row * N + col0);
#pragma unroll
        for (int i = 0; i < (EPI == CE_EPI_BIAS_RES16_F16 ? 4 : 0); ++i)
          rres[i] = row < M ? __ldg(rp + i) : make_uint4(0u, 0u, 0u, 0u);
      }
      mbar_wait(bar_acc_full + 8 * as, ((uint32_t)(t / kWsAcc)) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      uint32_t v[32];
      {
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BN + colgrp * 32);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
              "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
              "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
              "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
            : "r"(taddr)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      }
      // the accumulator stage is in registers now: hand it back to the MMA issuer before the stores
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_acc_empty + 8 * as);
      float f[32];
      if (kBiasRegs) {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]) + bias_r[kBiasRegs ? j : 0];
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]) + __shfl_sync(0xffffffffu, bias_lane, j);
      }
      if (EPI == CE_EPI_BIAS_RES16_F16) {
        // the fp32 sums acc + bias + residual are rounded ONCE, to the fp16 row that is staged and drained below
#pragma unroll
        for (int i = 0; i < (EPI == CE_EPI_BIAS_RES16_F16 ? 4 : 0); ++i) {
          const __half2* h = reinterpret_cast<const __half2*>(&rres[i]);
#pragma unroll
          for (int e2 = 0; e2 < 4; ++e2) {
            const float2 rf = __half22float2(h[e2]);
            f[8 * i + 2 * e2] += rf.x;
            f[8 * i + 2 * e2 + 1] += rf.y;
          }
        }
      }
      if (EPI == CE_EPI_BIAS_RES_F32) {
#pragma unroll 1
        for (int p2 = 0; p2 < 2; ++p2) {  // two passes of 16 fp32 columns (64 bytes per staged row)
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            float4 w;
            w.x = p2 ? f[16 + j + 0] : f[j + 0];
            w.y = p2 ? f[16 + j + 1] : f[j + 1];
            w.z = p2 ? f[16 + j + 2] : f[j + 2];
            w.w = p2 ? f[16 + j + 3] : f[j + 3];
            *reinterpret_cast<float4*>(st + (size_t)lane * kStageRow + (size_t)j * 4) = w;
          }
          __syncwarp();
          const int col = col0 + 16 * p2 + c16;
#pragma unroll 1
          for (int r0 = 0; r0 < 32; r0 += 16) {
            float res[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {  // eight independent residual loads in flight per lane
              const int row = row0 + r0 + 2 * u + sub;
              res[u] = row < M ? __ldg(residual + (size_t)row * N + col) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const int rr = r0 + 2 * u + sub, row = row0 + rr;
              const float x = *reinterpret_cast<const float*>(st + (size_t)rr * kStageRow + (size_t)c16 * 4);
              if (row < M) out32[(size_t)row * N + col] = x + res[u];
            }
          }
          __syncwarp();
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint4 pk;
          const __half2 h0 = act_pack<EPI>(f[j + 0], f[j + 1]), h1 = act_pack<EPI>(f[j + 2], f[j + 3]);
          const __half2 h2 = act_pack<EPI>(f[j + 4], f[j + 5]), h3 = act_pack<EPI>(f[j + 6], f[j + 7]);
          pk.x = *reinterpret_cast<const uint32_t*>(&h0);
          pk.y = *reinterpret_cast<const uint32_t*>(&h1);
          pk.z = *reinterpret_cast<const uint32_t*>(&h2);
          pk.w = *reinterpret_cast<const uint32_t*>(&h3);
          *reinterpret_cast<uint4*>(st + (size_t)lane * kStageRow + (size_t)j * 2) = pk;
        }
        __syncwarp();
        // drain: four 64-byte row segments (32 fp16 columns each) per instruction, 8 bytes per lane.  A half-warp reads
        // rows (r, r + 4): 4 x 80 B = 80 words = 16 mod 32, so its two 64-byte segments fall on disjoint banks.
        const int c8 = lane & 7, rsel = lane >> 3;
        const int rmap = (rsel & 1) * 4 + (rsel >> 1);   // {0, 4, 1, 5}
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int rr = (it >> 1) * 8 + (it & 1) * 2 + rmap, row = row0 + rr;
          if (row < M) {
            const uint2 x = *reinterpret_cast<const uint2*>(st + (size_t)rr * kStageRow + (size_t)c8 * 8);
            *reinterpret_cast<uint2*>(out16 + (size_t)row * N + col0 + 4 * c8) = x;
          }
        }
        __syncwarp();
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kWsAcc * BN) : "memory");
  }
}

template <int EPI, bool RESIDENT>
int launch_ws(const CUtensorMap& map_a, const CUtensorMap& map_w, int M, int N, int K, const float* bias,
              const float* residual, __half* out16, float* out32, cudaStream_t st, const int* m_dev) {
  const size_t extra = 1024 /*align*/ + 256 /*barriers*/ + (size_t)kWsEpiWarps * kStageWarpBytes;
  const size_t smem = RESIDENT ? (size_t)(K / BK) * kTileBBytes + (size_t)kWsStages * kTileABytes + extra
                               : (size_t)kWsStages * kStageBytes + extra;
  static size_t configured = 0;
  if (configured < smem) {
    SB_CUDA(cudaFuncSetAttribute(ce_gemm_ws_kernel<EPI, RESIDENT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int tiles = (N / BN) * ((M + BM - 1) / BM);
  const int grid = std::max(N / BN, std::min(sms, tiles));
  ce_gemm_ws_kernel<EPI, RESIDENT><<<grid, kWsThreads, smem, st>>>(map_a, map_w, M, N, K, bias, residual, out16, out32,
                                                                   m_dev);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

}  // namespace

// rows x cols fp16 row-major (cols contiguous) -> 2-D tensor map with a 64 x 128 box and 128-byte swizzle
int ce_make_tensor_map(CUtensorMap* map, const void* ptr, int64_t rows, int64_t cols) {
  EncodeTiledFn enc = get_encode();
  SB_REQUIRE(enc != nullptr, SB_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  SB_REQUIRE(cols % BK == 0, SB_ERR_ARG, "ce_gemm: K=%lld must be a multiple of %d", (long long)cols, BK);
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)BM};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SB_REQUIRE(r == CUDA_SUCCESS, SB_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return SB_OK;
}

int ce_gemm_launch(int epi, const CUtensorMap& map_a, const CUtensorMap& map_w, int M, int N, int K, const float* bias,
                   const float* residual, __half* out16, float* out32, cudaStream_t st, const int* m_dev) {
  SB_REQUIRE(N % BN == 0 && K % BK == 0, SB_ERR_ARG, "ce_gemm: N=%d / K=%d must be multiples of %d / %d", N, K, BN, BK);
  if ((M + BM - 1) / BM >= 4) {  // persistent kernels: weight-stationary when the weight tile fits, streaming otherwise
    if (K <= 384) {
      switch (epi) {
        case CE_EPI_BIAS_F16:
          return launch_ws<CE_EPI_BIAS_F16, true>(map_a, map_w, M, N, K, bias, residual, out16, out32, st, m_dev);
        case CE_EPI_BIAS_GELU_F16:
          return launch_ws<CE_EPI_BIAS_GELU_F16, true>(map_a, map_w, M, N, K, bias, residual, out16, out32, st, m_dev);
        case CE_EPI_BIAS_RES_F32:
          return launch_ws<CE_EPI_BIAS_RES_F32, true>(map_a, map_w, M, N, K, bias, residual, out16, out32, st, m_dev);
        case CE_EPI_BIAS_RES16_F16:
          return launch_ws<CE_EPI_BIAS_RES16_F16, true>(map_a, map_w, M, N, K, bias, residual, out16, out32, st, m_dev);
      }
    } else {
      switch (epi) {
        case CE_EPI_BIAS_F16:
          return launch_ws<CE_EPI_BIAS_F16, false>(map_a, map_w, M, N, K, bias, residual, out16, out32, st, m_dev);
        case CE_EPI_BIAS_GELU_F16:
          return launch_ws<CE_EPI_BIAS_GELU_F16, false>(map_a, map_w, M, N, K, bias, residual, out16, out32, st, m_dev);
        case CE_EPI_BIAS_RES_F32:
          return launch_ws<CE_EPI_BIAS_RES_F32, false>(map_a, map_w, M, N, K, bias, residual, out16, out32, st, m_dev);
        case CE_EPI_BIAS_RES16_F16:
          return launch_ws<CE_EPI_BIAS_RES16_F16, false>(map_a, map_w, M, N, K, bias, residual, out16, out32, st, m_dev);
      }
    }
  }
  dim3 grid(N / BN, (M + BM - 1) / BM);
  switch (epi) {
    case CE_EPI_BIAS_F16: {
      static bool once = false;
      if (!once) {
        SB_CUDA(cudaFuncSetAttribute(ce_gemm_kernel<CE_EPI_BIAS_F16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)kGemmSmem));
        once = true;
      }
      ce_gemm_kernel<CE_EPI_BIAS_F16><<<grid, kGemmThreads, kGemmSmem, st>>>(map_a, map_w, M, N, K, bias, residual,
                                                                             out16, out32, m_dev);
      break;
    }
    case CE_EPI_BIAS_GELU_F16: {
      static bool once = false;
      if (!once) {
        SB_CUDA(cudaFuncSetAttribute(ce_gemm_kernel<CE_EPI_BIAS_GELU_F16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)kGemmSmem));
        once = true;
      }
      ce_gemm_kernel<CE_EPI_BIAS_GELU_F16><<<grid, kGemmThreads, kGemmSmem, st>>>(map_a, map_w, M, N, K, bias, residual, out16, out32, m_dev);
      break;
    }
    case CE_EPI_BIAS_RES_F32: {
      static bool once = false;
      if (!once) {
        SB_CUDA(cudaFuncSetAttribute(ce_gemm_kernel<CE_EPI_BIAS_RES_F32>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)kGemmSmem));
        once = true;
      }
      ce_gemm_kernel<CE_EPI_BIAS_RES_F32><<<grid, kGemmThreads, kGemmSmem, st>>>(map_a, map_w, M, N, K, bias, residual,
                                                                                 out16, out32, m_dev);
      break;
    }
    case CE_EPI_BIAS_RES16_F16: {
      static bool once = false;
      if (!once) {
        SB_CUDA(cudaFuncSetAttribute(ce_gemm_kernel<CE_EPI_BIAS_RES16_F16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)kGemmSmem));
        once = true;
      }
      ce_gemm_kernel<CE_EPI_BIAS_RES16_F16><<<grid, kGemmThreads, kGemmSmem, st>>>(map_a, map_w, M, N, K, bias, residual,
                                                                                   out16, out32, m_dev);
      break;
    }
    default:
      sb_set_error("ce_gemm: unknown epilogue %d", epi);
      return SB_ERR_ARG;
  }
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}
