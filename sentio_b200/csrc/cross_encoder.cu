// cross_encoder.cu -- K5: BERT-style sequence classifier forward (MiniLM-L6 shape by default) for the reranker.
//
// Replaces the remote Jina rerank call behind JinaReranker.rerank (reference src/core/rerankers/jina_reranker.py:139-144).
// Per layer:  QKV GEMM (tcgen05, bias)  ->  masked softmax attention  ->  out-proj GEMM (+bias +residual, fp32)
//             -> LayerNorm -> FFN-up GEMM (+bias, erf-GELU) -> FFN-down GEMM (+bias +residual, fp32) -> LayerNorm.
// The residual stream stays fp32 in HBM; every GEMM operand is an fp16 copy written by the producing kernel; all GEMM
// accumulation is fp32 in tensor memory (ce_gemm.cu).
//
// PACKED TOKENS: positions beyond a pair's length are padding -- never read as keys (masked) and never consumed, which is
// what the additive -inf mask of the HuggingFace oracle yields for the [CLS] logit -- so they are not computed at all: the
// tokens of all pairs of a forward pass are packed back to back (pair p occupies rows [cu[p], cu[p] + len[p])), every
// GEMM / LayerNorm runs over sum(len) rows instead of P*S, attention only visits the key tiles below len.  The packed row
// count only exists on the device (cu[P]); grids are sized for P*S and the kernels clamp to it (ce_gemm.cuh m_dev), so
// the forward stays a pure enqueue with no host synchronisation.
//
// flops per pair = L * (24*len*H^2 + 4*len^2*H)  (2.87 GFLOP at L=6, H=384, len=S=128); bound: tensor pipe.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "ce_gemm.cuh"

struct CeLayer {
  __half *wqkv, *wo, *w1, *w2;            // fp16 GEMM weights: [3H,H] [H,H] [I,H] [H,I]
  float *bqkv, *bo, *b1, *b2;             // fp32 biases
  float *ln1_g, *ln1_b, *ln2_g, *ln2_b;   // fp32 LayerNorm parameters
  CUtensorMap m_wqkv, m_wo, m_w1, m_w2;
};

struct CeModel {
  sb_ce_config cfg;
  float *word_emb = nullptr, *pos_emb = nullptr, *type_emb = nullptr, *emb_ln_g = nullptr, *emb_ln_b = nullptr;
  float *pool_w = nullptr, *pool_b = nullptr, *cls_w = nullptr, *cls_b = nullptr;
  std::vector<CeLayer> layers;
  std::vector<void*> allocs;
  // activation workspace (grow-only), sized for m_cap rows
  int64_t m_cap = 0;
  float *x32 = nullptr, *pre32 = nullptr;          // residual stream, pre-LayerNorm sums  [M,H]
  __half* pre16 = nullptr;                         // pre-LayerNorm sums of the fp16 residual stream  [M,H]
  // fp16 residual stream (the reranker): x16 is BOTH the GEMM operand and the residual, the pre-LN sum is stored in fp16;
  // half the bytes of the two N = 384 GEMM epilogues and of the LayerNorms.  CPU study (oracle forward with the LayerNorm
  // inputs and outputs rounded to fp16): sigmoid scores move by 1.6e-4 relative (tolerance 1e-3).  The embedder keeps the
  // fp32 stream: its output is the hidden state itself, compared element-wise.
  bool fp16_stream = false;
  __half *x16 = nullptr, *qkv16 = nullptr, *ctx16 = nullptr, *ffn16 = nullptr;  // [M,H] [M,3H] [M,H] [M,I]
  CUtensorMap m_x16, m_ctx16, m_ffn16;
  std::vector<void*> act_allocs;
  int32_t* cu = nullptr;   // [cu_cap + 1] first packed row of every pair; cu[P] = packed row count of the pass
  int64_t cu_cap = 0;
  unsigned long long* stats = nullptr;  // device: {pairs, sum len, sum len^2} since the last reset (sb_ce_stats)
  // last layer: only the [CLS] row of a pair reaches the head -> P-row buffers for everything after its K/V projection
  float *xcls32 = nullptr, *precls32 = nullptr;                       // [P,H]
  __half *xcls16 = nullptr, *ctxcls16 = nullptr, *ffncls16 = nullptr;  // [P,H] [P,H] [P,I]
  CUtensorMap m_xcls16, m_ctxcls16, m_ffncls16;
  std::vector<void*> cls_allocs;
  // embedder use (sb_enc_*): optional output projection of the final [CLS] state, fp32 [out_dim, H] + [out_dim]
  float *proj_w = nullptr, *proj_b = nullptr;
  int out_dim = 0;
};

// Per-shard store of pre-tokenised documents for the batched rerank path: doc i -> tok[i][0..len[i])
struct CeDocTokens {
  uint16_t* tok = nullptr;   // [n][ld]
  int32_t* len = nullptr;    // [n]
  int64_t n = 0, id_base = 0;
  int32_t ld = 0;
};

void ce_tokens_free(CeDocTokens* t) {
  if (!t) return;
  if (t->tok) cudaFree(t->tok);
  if (t->len) cudaFree(t->len);
  delete t;
}

void ce_model_free(CeModel* m) {
  if (!m) return;
  for (void* p : m->allocs) cudaFree(p);
  for (void* p : m->act_allocs) cudaFree(p);
  if (m->cu) cudaFree(m->cu);
  if (m->stats) cudaFree(m->stats);
  for (void* p : m->cls_allocs) cudaFree(p);
  delete m;
}

namespace {

// ------------------------------------------------------------------------------------------------ small kernels
__global__ void f32_to_f16_kernel(const float* __restrict__ in, __half* __restrict__ out, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __float2half_rn(in[i]);
}

// cu[p] = sum_{i<p} clamp(len[i], 1, S): first packed row of pair p; cu[P] = packed row count.  One CTA.
__global__ void __launch_bounds__(1024) ce_cu_kernel(const int32_t* __restrict__ lens, int P, int S,
                                                     int32_t* __restrict__ cu, unsigned long long* __restrict__ stats) {
  __shared__ int warp_sum[32];
  __shared__ int carry_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int base = 0; base < P; base += 1024) {
    const int i = base + tid;
    const int v = i < P ? min(max(lens[i], 1), S) : 0;
    int x = v;
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_sum[warp] = x;
    __syncthreads();
    if (warp == 0) {
      int w = warp_sum[lane];
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += y;
      }
      warp_sum[lane] = w;  // inclusive
    }
    __syncthreads();
    const int carry = carry_s;
    const int excl = carry + (warp ? warp_sum[warp - 1] : 0) + x - v;
    if (i < P) cu[i] = excl;
    {
      unsigned long long sq = (unsigned long long)v * (unsigned long long)v;
      for (int o = 16; o; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
      if (lane == 0 && sq) atomicAdd(stats + 2, sq);
    }
    __syncthreads();
    if (tid == 1023) carry_s = carry + warp_sum[31];
    __syncthreads();
  }
  if (tid == 0) {
    cu[P] = carry_s;
    atomicAdd(stats + 0, (unsigned long long)P);
    atomicAdd(stats + 1, (unsigned long long)carry_s);
  }
}

// One warp per (pair, position): x = LN(word[id] + pos[s] + type[tt]); writes the fp32 residual and its fp16 GEMM copy
// to the PACKED row cu[pair] + s.  M = P * S padded positions are enumerated, positions >= len produce nothing.
template <int H>
__global__ void ce_embed_ln_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ tts,
                                   const int32_t* __restrict__ lens, const int32_t* __restrict__ cu, int M, int S,
                                   int vocab, int type_vocab, const float* __restrict__ word,
                                   const float* __restrict__ pos, const float* __restrict__ type,
                                   const float* __restrict__ g, const float* __restrict__ b, float eps,
                                   float* __restrict__ x32, __half* __restrict__ x16) {
  constexpr int PER = H / 32;
  const int prow = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (prow >= M) return;
  const int pair = prow / S, s = prow % S;
  if (s >= min(max(lens[pair], 1), S)) return;
  const int row = cu[pair] + s;
  int id = ids[prow], tt = tts[prow];
  id = min(max(id, 0), vocab - 1);
  tt = min(max(tt, 0), type_vocab - 1);
  float v[PER];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    const int c = lane + 32 * i;
    v[i] = word[(size_t)id * H + c] + pos[(size_t)s * H + c] + type[(size_t)tt * H + c];
    sum += v[i];
  }
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum / H;
  float var = 0.f;
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    const float d = v[i] - mean;
    var += d * d;
  }
  for (int o = 16; o; o >>= 1) var += __shfl_xor_sync(0xffffffffu, var, o);
  const float rstd = rsqrtf(var / H + eps);
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    const int c = lane + 32 * i;
    const float y = (v[i] - mean) * rstd * g[c] + b[c];
    if (x32) x32[(size_t)row * H + c] = y;
    x16[(size_t)row * H + c] = __float2half_rn(y);
  }
}

__device__ __forceinline__ float ln_load(const float* p) { return *p; }
__device__ __forceinline__ float ln_load(const __half* p) { return __half2float(*p); }

// LayerNorm of the pre-LN sum (fp32, or fp16 on the fp16 residual stream) -> fp16 GEMM copy (+ the fp32 residual when
// x32 != NULL).  A warp normalises kLnRows CONSECUTIVE rows: all of their loads are issued before the first reduction, so
// four rows' worth of memory latency overlap (one row per warp was latency bound: 48 us for 142 k rows, 3.4 TB/s).  Lane l
// owns the PER = H / 32 contiguous columns [l * PER, (l + 1) * PER) of each row (8-byte / 16-byte accesses).
constexpr int kLnRows = 4;
template <int H, typename TIn>
__global__ void ce_ln_kernel(const TIn* __restrict__ pre, int M_host, const int32_t* __restrict__ m_dev,
                             const float* __restrict__ g, const float* __restrict__ b, float eps,
                             float* __restrict__ x32, __half* __restrict__ x16) {
  constexpr int PER = H / 32;
  static_assert(PER % 4 == 0, "hidden size must be a multiple of 128");
  const int row0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * kLnRows, lane = threadIdx.x & 31;
  const int M = m_dev ? __ldg(m_dev) : M_host;
  if (row0 >= M) return;
  float v[kLnRows][PER];
#pragma unroll
  for (int r = 0; r < kLnRows; ++r) {
    const size_t base = (size_t)min(row0 + r, M - 1) * H + (size_t)lane * PER;   // rows beyond M: re-read the last one
#pragma unroll
    for (int i = 0; i < PER; i += 4) {
      if constexpr (sizeof(TIn) == 2) {
        const uint2 raw = *reinterpret_cast<const uint2*>(pre + base + i);
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
        const float2 c = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
        v[r][i] = a.x; v[r][i + 1] = a.y; v[r][i + 2] = c.x; v[r][i + 3] = c.y;
      } else {
        const float4 raw = *reinterpret_cast<const float4*>(pre + base + i);
        v[r][i] = raw.x; v[r][i + 1] = raw.y; v[r][i + 2] = raw.z; v[r][i + 3] = raw.w;
      }
    }
  }
  float mean[kLnRows], rstd[kLnRows];
#pragma unroll
  for (int r = 0; r < kLnRows; ++r) {
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < PER; i += 4) sum += (v[r][i] + v[r][i + 1]) + (v[r][i + 2] + v[r][i + 3]);
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    mean[r] = sum / H;
    float var = 0.f;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const float d = v[r][i] - mean[r];
      var += d * d;
    }
    for (int o = 16; o; o >>= 1) var += __shfl_xor_sync(0xffffffffu, var, o);
    rstd[r] = rsqrtf(var / H + eps);
  }
#pragma unroll
  for (int i = 0; i < PER; i += 4) {
    const int c = lane * PER + i;
    const float4 gg = *reinterpret_cast<const float4*>(g + c), bb = *reinterpret_cast<const float4*>(b + c);
#pragma unroll
    for (int r = 0; r < kLnRows; ++r) {
      if (row0 + r >= M) break;
      const size_t base = (size_t)(row0 + r) * H + (size_t)c;
      float4 y;
      y.x = (v[r][i] - mean[r]) * rstd[r] * gg.x + bb.x;
      y.y = (v[r][i + 1] - mean[r]) * rstd[r] * gg.y + bb.y;
      y.z = (v[r][i + 2] - mean[r]) * rstd[r] * gg.z + bb.z;
      y.w = (v[r][i + 3] - mean[r]) * rstd[r] * gg.w + bb.w;
      if (x32) *reinterpret_cast<float4*>(x32 + base) = y;
      const __half2 h0 = __floats2half2_rn(y.x, y.y), h1 = __floats2half2_rn(y.z, y.w);
      uint2 pk;
      pk.x = *reinterpret_cast<const uint32_t*>(&h0);
      pk.y = *reinterpret_cast<const uint32_t*>(&h1);
      *reinterpret_cast<uint2*>(x16 + base) = pk;
    }
  }
}

// Long-sequence fallback (S > 256): masked softmax attention, one CTA per (pair, head), one thread per query row; K/V of the head staged in smem as fp32.
// Single pass online softmax (running max / sum), scores never leave registers.
template <int DH>
__global__ void __launch_bounds__(128) ce_attention_kernel(const __half* __restrict__ qkv, const int32_t* __restrict__ lengths,
                                                           const int32_t* __restrict__ cu, int S, int H, int heads,
                                                           __half* __restrict__ ctx) {
  extern __shared__ float att_sm[];
  const int pair = blockIdx.x / heads, head = blockIdx.x % heads;
  const int len = min(max(lengths[pair], 1), S);
  float* Ks = att_sm;                 // [S][DH]
  float* Vs = att_sm + (size_t)S * DH;
  const size_t row0 = (size_t)cu[pair];
  const int ld = 3 * H;
  for (int i = threadIdx.x; i < len * (DH / 2); i += blockDim.x) {
    const int j = i / (DH / 2), c = (i % (DH / 2)) * 2;
    const __half2 kk = *reinterpret_cast<const __half2*>(qkv + (row0 + j) * ld + H + head * DH + c);
    const __half2 vv = *reinterpret_cast<const __half2*>(qkv + (row0 + j) * ld + 2 * H + head * DH + c);
    const float2 kf = __half22float2(kk), vf = __half22float2(vv);
    Ks[j * DH + c] = kf.x; Ks[j * DH + c + 1] = kf.y;
    Vs[j * DH + c] = vf.x; Vs[j * DH + c + 1] = vf.y;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < len; i += blockDim.x) {
    __half* out = ctx + (row0 + i) * H + head * DH;
    float q[DH];
    const float scale = rsqrtf((float)DH);
#pragma unroll
    for (int c = 0; c < DH; c += 2) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(qkv + (row0 + i) * ld + head * DH + c));
      q[c] = f.x * scale;
      q[c + 1] = f.y * scale;
    }
    float m = -INFINITY, l = 0.f, acc[DH];
#pragma unroll
    for (int c = 0; c < DH; ++c) acc[c] = 0.f;
    for (int j = 0; j < len; ++j) {
      float s = 0.f;
#pragma unroll
      for (int c = 0; c < DH; ++c) s = fmaf(q[c], Ks[j * DH + c], s);
      if (s > m) {
        const float corr = __expf(m - s);
        l *= corr;
#pragma unroll
        for (int c = 0; c < DH; ++c) acc[c] *= corr;
        m = s;
      }
      const float pj = __expf(s - m);
      l += pj;
#pragma unroll
      for (int c = 0; c < DH; ++c) acc[c] = fmaf(pj, Vs[j * DH + c], acc[c]);
    }
    const float inv = 1.f / l;
#pragma unroll
    for (int c = 0; c < DH; c += 2)
      *reinterpret_cast<__half2*>(out + c) = __floats2half2_rn(acc[c] * inv, acc[c + 1] * inv);
  }
}

// Masked softmax attention on the tensor cores.  One CTA per (pair, head), 4 warps x S_MAX / 64 query tiles of 16 rows; the head's K and V
// (S x 32 fp16) are staged in shared memory (rows padded to 80 B: conflict-free fragment loads / ldmatrix), scores
// S = Q K^T and O = P V are mma.sync.m16n8k16 (fp16 in, fp32 accumulate), the softmax runs on the accumulator fragments
// in registers and the probabilities are re-used directly as the A operand of the second product (no smem round trip).
// Packed layout: the pair's rows are [cu[pair], cu[pair] + len); key tiles at or beyond len are skipped.
__device__ __forceinline__ void mma_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// HPC = heads of one pair handled by a CTA, one after the other: while head h is being computed the K/V rows of head
// h + 1 stream into the second shared-memory buffer with cp.async, so only the first head of a CTA waits for its operands
// (run 16's profile: a third of all stall samples sat on the K/V staging of one-head CTAs).
template <int S_MAX, int HPC>
__global__ void __launch_bounds__(128, S_MAX > 128 ? 2 : 4) ce_attention_mma_kernel(const __half* __restrict__ qkv,
                                                                const int32_t* __restrict__ lengths,
                                                                const int32_t* __restrict__ cu, int S, int H,
                                                                int heads, __half* __restrict__ ctx) {
  constexpr int DH = 32, LDS_ROW = 40;  // halves per padded smem row (80 B)
  constexpr int NT = S_MAX / 8;         // key tiles of 8
  constexpr int MT = S_MAX / 64;        // 16-row query tiles per warp (4 warps cover S_MAX rows)
  constexpr int NBUF = HPC > 1 ? 2 : 1;
  __shared__ __align__(16) __half Ks_all[NBUF][S_MAX * LDS_ROW];
  __shared__ __align__(16) __half Vs_all[NBUF][S_MAX * LDS_ROW];
  const int groups = heads / HPC;
  const int pair = blockIdx.x / groups, head0 = (blockIdx.x % groups) * HPC;
  const int len = min(min(max(lengths[pair], 1), S), S_MAX);
  const size_t row0 = (size_t)cu[pair];
  const int ld = 3 * H;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  // 16-row query tiles are dealt round-robin (tile j -> warp j & 3): a pair of ~90 tokens has 6 tiles, so every warp
  // has work (the contiguous 32-rows-per-warp split left warp 3 idle for every pair shorter than 97 tokens).  Rotating
  // the assignment per CTA to spread the two-tile warps over the SM's four schedulers was measured and changes nothing
  // (2741 vs 2749 queries/s, profiles/r02_run12_ab_ce_{base,norot}.json).
  const int vwarp = warp;
  const int stage_rows = min(S_MAX, (len + 31) & ~31);  // 32-key groups beyond len are never touched
  // rows [len, stage_rows) are masked keys: zeros (finite products), written once -- len belongs to the pair, not the head
  const int zero_slots = (stage_rows - len) * 4;
  for (int i = tid; i < zero_slots * NBUF; i += 128) {
    const int bsel = i / zero_slots, r = i % zero_slots;
    const int j = len + (r >> 2), c = (r & 3) * 8;
    *reinterpret_cast<uint4*>(&Ks_all[bsel][j * LDS_ROW + c]) = make_uint4(0u, 0u, 0u, 0u);
    *reinterpret_cast<uint4*>(&Vs_all[bsel][j * LDS_ROW + c]) = make_uint4(0u, 0u, 0u, 0u);
  }
  auto stage = [&](int bsel, int head) {
    for (int i = tid; i < len * 4; i += 128) {
      const int j = i >> 2, c = (i & 3) * 8;
      cp_async16(smem_u32(&Ks_all[bsel][j * LDS_ROW + c]), qkv + (row0 + j) * ld + H + head * DH + c);
      cp_async16(smem_u32(&Vs_all[bsel][j * LDS_ROW + c]), qkv + (row0 + j) * ld + 2 * H + head * DH + c);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  stage(0, head0);
  // softmax in base 2: scores are scaled by log2(e) / sqrt(d_head) once, the exponentials are bare ex2
  const float scale = rsqrtf((float)DH) * 1.4426950408889634f;
#pragma unroll 1
  for (int hh = 0; hh < HPC; ++hh) {
  const int head = head0 + hh;
  const __half* Ks = Ks_all[hh % NBUF];
  const __half* Vs = Vs_all[hh % NBUF];
  // Q fragments (A operand): rows g / g+8 of a 16-row tile, two k-steps of 16 columns (2t.. and 2t+8..)
  auto load_q = [&](uint32_t (&qa)[2][4], int r0) {
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      const __half* qlo = qkv + (row0 + min(r0 + g, len - 1)) * ld + head * DH + ks * 16 + 2 * t;
      const __half* qhi = qkv + (row0 + min(r0 + g + 8, len - 1)) * ld + head * DH + ks * 16 + 2 * t;
      qa[ks][0] = *reinterpret_cast<const uint32_t*>(qlo);
      qa[ks][1] = *reinterpret_cast<const uint32_t*>(qhi);
      qa[ks][2] = *reinterpret_cast<const uint32_t*>(qlo + 8);
      qa[ks][3] = *reinterpret_cast<const uint32_t*>(qhi + 8);
    }
  };
  // the first two tiles of this warp are fetched before waiting for K/V so the global round trips overlap (all the tiles
  // there are when S_MAX = 128; the S_MAX = 256 variant fetches tiles 2, 3 inside the loop)
  uint32_t qa_all[2][2][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) load_q(qa_all[mt], (mt * 4 + vwarp) * 16);
  if (hh + 1 < HPC) {  // next head's K/V into the other buffer (its last readers passed the barrier that ended hh - 1)
    stage((hh + 1) % NBUF, head + 1);
    asm volatile("cp.async.wait_group 1;" ::: "memory");
  } else {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  }
  __syncthreads();
#pragma unroll 1
  for (int mt = 0; mt < MT; ++mt) {
    const int r0 = (mt * 4 + vwarp) * 16;  // first query row of this 16-row tile
    if (r0 >= len) break;                  // no such rows in the packed layout
    __half* out_lo = ctx + (row0 + r0 + g) * H + head * DH;
    __half* out_hi = ctx + (row0 + r0 + g + 8) * H + head * DH;
    uint32_t qa[2][4];
    if (mt < 2) {
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int e = 0; e < 4; ++e) qa[ks][e] = mt ? qa_all[1][ks][e] : qa_all[0][ks][e];
    } else {
      load_q(qa, r0);
    }
    float sc[NT][4];
#pragma unroll
    for (int nc = 0; nc < NT / 4; ++nc) {  // groups of 32 keys: 8 independent MMAs per branch keep the tensor pipe fed
#pragma unroll
      for (int i = 0; i < 4; ++i) sc[nc * 4 + i][0] = sc[nc * 4 + i][1] = sc[nc * 4 + i][2] = sc[nc * 4 + i][3] = 0.f;
      if (nc * 32 < len) {  // CTA-uniform: groups at or beyond len are entirely masked
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int nt = nc * 4 + i;
            const __half* kp = Ks + (nt * 8 + g) * LDS_ROW + ks * 16 + 2 * t;
            mma_16816(sc[nt], qa[ks], *reinterpret_cast<const uint32_t*>(kp), *reinterpret_cast<const uint32_t*>(kp + 8));
          }
        }
      }
    }
    // masked softmax over the keys; a row's values live in the 4 lanes sharing g.  Work is skipped per 32-key group
    // (CTA-uniform): groups at or beyond len hold no keys (their probabilities are never read by the P V loop below) and
    // only the group that straddles len needs the per-key mask.  The maximum is taken on the raw scores (scale > 0) and
    // the scale folded into the exponent: p = ex2(s * scale - m * scale), one FFMA per score.
    float mlo = -INFINITY, mhi = -INFINITY;
#pragma unroll
    for (int nc = 0; nc < NT / 4; ++nc) {
      if (nc * 32 < len) {
        if (nc * 32 + 32 > len) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int nt = nc * 4 + i, key = nt * 8 + 2 * t;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              if (key + e >= len) sc[nt][e] = sc[nt][2 + e] = -INFINITY;
            }
          }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int nt = nc * 4 + i;
          mlo = fmaxf(mlo, fmaxf(sc[nt][0], sc[nt][1]));
          mhi = fmaxf(mhi, fmaxf(sc[nt][2], sc[nt][3]));
        }
      }
    }
    mlo = fmaxf(mlo, __shfl_xor_sync(0xffffffffu, mlo, 1));
    mlo = fmaxf(mlo, __shfl_xor_sync(0xffffffffu, mlo, 2));
    mhi = fmaxf(mhi, __shfl_xor_sync(0xffffffffu, mhi, 1));
    mhi = fmaxf(mhi, __shfl_xor_sync(0xffffffffu, mhi, 2));
    const float nlo = -mlo * scale, nhi = -mhi * scale;
    float llo = 0.f, lhi = 0.f;
#pragma unroll
    for (int nc = 0; nc < NT / 4; ++nc) {
      if (nc * 32 < len) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int nt = nc * 4 + i;
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            sc[nt][e] = ex2_approx(fmaf(sc[nt][e], scale, nlo));
            sc[nt][2 + e] = ex2_approx(fmaf(sc[nt][2 + e], scale, nhi));
            llo += sc[nt][e];
            lhi += sc[nt][2 + e];
          }
        }
      }
    }
    llo += __shfl_xor_sync(0xffffffffu, llo, 1);
    llo += __shfl_xor_sync(0xffffffffu, llo, 2);
    lhi += __shfl_xor_sync(0xffffffffu, lhi, 1);
    lhi += __shfl_xor_sync(0xffffffffu, lhi, 2);
    // O = P V : P fragments come straight from the score accumulators, V fragments via ldmatrix.trans
    float oc[DH / 8][4];
#pragma unroll
    for (int n = 0; n < DH / 8; ++n) oc[n][0] = oc[n][1] = oc[n][2] = oc[n][3] = 0.f;
#pragma unroll
    for (int kk = 0; kk < NT / 2; ++kk) {
      if ((kk >> 1) * 32 >= len) continue;  // 32-key group entirely beyond len: its probabilities are exactly 0
      uint32_t pa[4];
      pa[0] = pack_h2(sc[2 * kk][0], sc[2 * kk][1]);
      pa[1] = pack_h2(sc[2 * kk][2], sc[2 * kk][3]);
      pa[2] = pack_h2(sc[2 * kk + 1][0], sc[2 * kk + 1][1]);
      pa[3] = pack_h2(sc[2 * kk + 1][2], sc[2 * kk + 1][3]);
#pragma unroll
      for (int n = 0; n < DH / 8; ++n) {
        uint32_t b0, b1;
        const uint32_t addr = smem_u32(Vs + (kk * 16 + (lane & 15)) * LDS_ROW + n * 8);
        asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0, %1}, [%2];" : "=r"(b0), "=r"(b1) : "r"(addr));
        mma_16816(oc[n], pa, b0, b1);
      }
    }
    const float ilo = 1.f / llo, ihi = 1.f / lhi;
#pragma unroll
    for (int n = 0; n < DH / 8; ++n) {
      if (r0 + g < len) *reinterpret_cast<uint32_t*>(out_lo + n * 8 + 2 * t) = pack_h2(oc[n][0] * ilo, oc[n][1] * ilo);
      if (r0 + g + 8 < len) *reinterpret_cast<uint32_t*>(out_hi + n * 8 + 2 * t) = pack_h2(oc[n][2] * ihi, oc[n][3] * ihi);
    }
  }
  __syncthreads();  // every warp is done with this head's buffer before it is refilled
  }
}

// Last layer: the head only consumes the [CLS] row of every pair, so attention is evaluated for that single query row.
// One warp per (pair, head): lane j scores keys j, j + 32, ... (fp32 dot over the 32 head dims), warp softmax, then lane c
// accumulates output dim c over all keys.  The warp also gathers its 32 columns of the pair's fp32 residual row into
// xcls32, the residual operand of the P-row out-projection that follows.
__global__ void __launch_bounds__(128) ce_attention_cls_kernel(const __half* __restrict__ qkv,
                                                                const int32_t* __restrict__ lengths,
                                                                const int32_t* __restrict__ cu, int P, int S, int H,
                                                                int heads, const float* __restrict__ x32,
                                                                const __half* __restrict__ x16,
                                                                __half* __restrict__ ctx_cls, float* __restrict__ xcls32) {
  constexpr int DH = 32, KPL = 16;  // keys per lane: S <= 512
  const int wg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (wg >= P * heads) return;
  const int pair = wg / heads, head = wg % heads;
  const int len = min(max(lengths[pair], 1), S);
  const size_t row0 = (size_t)cu[pair];
  const int ld = 3 * H;
  const float qmine = __half2float(qkv[row0 * ld + head * DH + lane]) * rsqrtf((float)DH);
  float qv[DH];
#pragma unroll
  for (int c = 0; c < DH; ++c) qv[c] = __shfl_sync(0xffffffffu, qmine, c);
  float sc[KPL];
  float mx = -INFINITY;
#pragma unroll
  for (int u = 0; u < KPL; ++u) {
    const int j = u * 32 + lane;
    sc[u] = -INFINITY;
    if (u * 32 < len && j < len) {
      const uint4* kp = reinterpret_cast<const uint4*>(qkv + (row0 + j) * ld + H + head * DH);
      float s = 0.f;
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const uint4 raw = __ldg(kp + v);
        const __half2* h = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = __half22float2(h[e]);
          s = fmaf(qv[v * 8 + 2 * e], f.x, s);
          s = fmaf(qv[v * 8 + 2 * e + 1], f.y, s);
        }
      }
      sc[u] = s;
      mx = fmaxf(mx, s);
    }
  }
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float l = 0.f;
#pragma unroll
  for (int u = 0; u < KPL; ++u) {
    sc[u] = (u * 32 < len && u * 32 + lane < len) ? __expf(sc[u] - mx) : 0.f;
    l += sc[u];
  }
  for (int o = 16; o; o >>= 1) l += __shfl_xor_sync(0xffffffffu, l, o);
  float acc = 0.f;
#pragma unroll
  for (int u = 0; u < KPL; ++u) {
    if (u * 32 >= len) break;  // warp-uniform
    const int nk = min(32, len - u * 32);
#pragma unroll 8
    for (int jj = 0; jj < nk; ++jj) {
      const float pj = __shfl_sync(0xffffffffu, sc[u], jj);
      acc = fmaf(pj, __half2float(qkv[(row0 + u * 32 + jj) * ld + 2 * H + head * DH + lane]), acc);
    }
  }
  ctx_cls[(size_t)pair * H + head * DH + lane] = __float2half_rn(acc / l);
  // the [CLS] row of the residual stream (fp32 stream, or the fp16 stream widened: the P-row tail of the last layer is fp32)
  xcls32[(size_t)pair * H + head * DH + lane] =
      x32 ? x32[row0 * H + head * DH + lane] : __half2float(x16[row0 * H + head * DH + lane]);
}

// pooled = tanh(Wp x_cls + bp); logit = w . pooled + b; relevance = sigmoid(logit).  fp32 throughout.
// One CTA per kHeadPairs pairs: every row of the pooler weight is read once per CTA and dotted with all of its pairs'
// [CLS] rows (one CTA per pair re-read the 590 KB matrix P times).
constexpr int kHeadPairs = 8;
__global__ void __launch_bounds__(512) ce_head_kernel(const float* __restrict__ x32, const int32_t* __restrict__ cu, int P,
                                                      int H, const float* __restrict__ pool_w,
                                                      const float* __restrict__ pool_b, const float* __restrict__ cls_w,
                                                      const float* __restrict__ cls_b, float* __restrict__ logits,
                                                      float* __restrict__ sig) {
  extern __shared__ float head_sm[];  // x_cls[kHeadPairs][H], partial[warps][kHeadPairs]
  const int pair0 = blockIdx.x * kHeadPairs, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int np = min(kHeadPairs, P - pair0);
  for (int i = threadIdx.x; i < kHeadPairs * H; i += blockDim.x) {
    const int q = i / H, c = i % H;
    // the pair's [CLS] row (cu == NULL: x32 is [P,H])
    head_sm[i] = q < np ? x32[(size_t)(cu ? cu[pair0 + q] : pair0 + q) * H + c] : 0.f;
  }
  __syncthreads();
  float part[kHeadPairs];
#pragma unroll
  for (int q = 0; q < kHeadPairs; ++q) part[q] = 0.f;
  for (int j = warp; j < H; j += nw) {
    float s[kHeadPairs];
#pragma unroll
    for (int q = 0; q < kHeadPairs; ++q) s[q] = 0.f;
    for (int c = lane; c < H; c += 32) {
      const float wv = pool_w[(size_t)j * H + c];
#pragma unroll
      for (int q = 0; q < kHeadPairs; ++q) s[q] = fmaf(wv, head_sm[q * H + c], s[q]);
    }
    const float cw = cls_w[j], pb = pool_b[j];
#pragma unroll
    for (int q = 0; q < kHeadPairs; ++q) {
      float v = s[q];
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      part[q] += cw * tanhf(v + pb);
    }
  }
  float* partial = head_sm + kHeadPairs * H;
  if (lane == 0)
#pragma unroll
    for (int q = 0; q < kHeadPairs; ++q) partial[warp * kHeadPairs + q] = part[q];
  __syncthreads();
  if (threadIdx.x < np) {
    float z = cls_b[0];
    for (int w = 0; w < nw; ++w) z += partial[w * kHeadPairs + threadIdx.x];
    logits[pair0 + threadIdx.x] = z;
    sig[pair0 + threadIdx.x] = 1.f / (1.f + expf(-z));
  }
}

int dev_alloc(std::vector<void*>& pool, void** out, size_t bytes) {
  SB_CUDA(cudaMalloc(out, bytes ? bytes : 16));
  pool.push_back(*out);
  return SB_OK;
}

int upload_f32(CeModel* m, const float*& src, float** dst, size_t n, cudaStream_t st) {
  int rc = dev_alloc(m->allocs, reinterpret_cast<void**>(dst), n * 4);
  if (rc) return rc;
  SB_CUDA(cudaMemcpyAsync(*dst, src, n * 4, cudaMemcpyHostToDevice, st));
  src += n;
  return SB_OK;
}

// upload fp32 host rows to a staging buffer and convert into an fp16 device matrix at dst (+row offset)
int upload_f16(sb_ctx* ctx, const float*& src, __half* dst, size_t n, cudaStream_t st) {
  int rc = ctx->misc_dev.reserve(n * 4);
  if (rc) return rc;
  SB_CUDA(cudaStreamSynchronize(st));  // staging buffer reuse
  SB_CUDA(cudaMemcpyAsync(ctx->misc_dev.p, src, n * 4, cudaMemcpyHostToDevice, st));
  f32_to_f16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ctx->misc_dev.as<float>(), dst, (int64_t)n);
  SB_CUDA(cudaGetLastError());
  src += n;
  return SB_OK;
}

int ensure_workspace(CeModel* m, int64_t P, int64_t M, cudaStream_t st) {
  if (!m->stats) {
    SB_CUDA(cudaMalloc(&m->stats, 3 * sizeof(unsigned long long)));
    SB_CUDA(cudaMemsetAsync(m->stats, 0, 3 * sizeof(unsigned long long), st));
  }
  if (P > m->cu_cap) {
    cudaDeviceSynchronize();
    if (m->cu) cudaFree(m->cu);
    m->cu = nullptr;
    m->cu_cap = 0;
    SB_CUDA(cudaMalloc(&m->cu, (size_t)(P + P / 4 + 2) * 4));
    m->cu_cap = P + P / 4 + 1;
    for (void* p : m->cls_allocs) cudaFree(p);
    m->cls_allocs.clear();
    const int64_t Pp = (m->cu_cap + 127) / 128 * 128;
    const int Hc = m->cfg.hidden, Ic = m->cfg.intermediate;
    int rc;
    if ((rc = dev_alloc(m->cls_allocs, (void**)&m->xcls32, (size_t)Pp * Hc * 4))) return rc;
    if ((rc = dev_alloc(m->cls_allocs, (void**)&m->precls32, (size_t)Pp * Hc * 4))) return rc;
    if ((rc = dev_alloc(m->cls_allocs, (void**)&m->xcls16, (size_t)Pp * Hc * 2))) return rc;
    if ((rc = dev_alloc(m->cls_allocs, (void**)&m->ctxcls16, (size_t)Pp * Hc * 2))) return rc;
    if ((rc = dev_alloc(m->cls_allocs, (void**)&m->ffncls16, (size_t)Pp * Ic * 2))) return rc;
    SB_CUDA(cudaMemsetAsync(m->xcls32, 0, (size_t)Pp * Hc * 4, st));
    SB_CUDA(cudaMemsetAsync(m->xcls16, 0, (size_t)Pp * Hc * 2, st));
    SB_CUDA(cudaMemsetAsync(m->ctxcls16, 0, (size_t)Pp * Hc * 2, st));
    SB_CUDA(cudaMemsetAsync(m->ffncls16, 0, (size_t)Pp * Ic * 2, st));
    if ((rc = ce_make_tensor_map(&m->m_xcls16, m->xcls16, Pp, Hc))) return rc;
    if ((rc = ce_make_tensor_map(&m->m_ctxcls16, m->ctxcls16, Pp, Hc))) return rc;
    if ((rc = ce_make_tensor_map(&m->m_ffncls16, m->ffncls16, Pp, Ic))) return rc;
  }
  const int64_t Mp = (M + 127) / 128 * 128;
  if (Mp <= m->m_cap) return SB_OK;
  cudaDeviceSynchronize();
  for (void* p : m->act_allocs) cudaFree(p);
  m->act_allocs.clear();
  m->m_cap = 0;
  const int H = m->cfg.hidden, I = m->cfg.intermediate;
  int rc;
  if ((rc = dev_alloc(m->act_allocs, (void**)&m->x32, (size_t)Mp * H * 4))) return rc;
  if ((rc = dev_alloc(m->act_allocs, (void**)&m->pre32, (size_t)Mp * H * 4))) return rc;
  if ((rc = dev_alloc(m->act_allocs, (void**)&m->pre16, (size_t)Mp * H * 2))) return rc;
  if ((rc = dev_alloc(m->act_allocs, (void**)&m->x16, (size_t)Mp * H * 2))) return rc;
  if ((rc = dev_alloc(m->act_allocs, (void**)&m->qkv16, (size_t)Mp * 3 * H * 2))) return rc;
  if ((rc = dev_alloc(m->act_allocs, (void**)&m->ctx16, (size_t)Mp * H * 2))) return rc;
  if ((rc = dev_alloc(m->act_allocs, (void**)&m->ffn16, (size_t)Mp * I * 2))) return rc;
  // padding rows of the GEMM A operands must be finite; stream-ordered with the forward pass that follows
  SB_CUDA(cudaMemsetAsync(m->x16, 0, (size_t)Mp * H * 2, st));
  SB_CUDA(cudaMemsetAsync(m->ctx16, 0, (size_t)Mp * H * 2, st));
  SB_CUDA(cudaMemsetAsync(m->ffn16, 0, (size_t)Mp * I * 2, st));
  SB_CUDA(cudaMemsetAsync(m->x32, 0, (size_t)Mp * H * 4, st));
  if ((rc = ce_make_tensor_map(&m->m_x16, m->x16, Mp, H))) return rc;
  if ((rc = ce_make_tensor_map(&m->m_ctx16, m->ctx16, Mp, H))) return rc;
  if ((rc = ce_make_tensor_map(&m->m_ffn16, m->ffn16, Mp, I))) return rc;
  m->m_cap = Mp;
  return SB_OK;
}

template <int H>
int ce_forward(sb_ctx* ctx, CeModel* m, const int32_t* ids, const int32_t* tts, const int32_t* lens, int P, int S,
               float* logits, float* sig, float* cls_out, cudaStream_t st) {
  const sb_ce_config& c = m->cfg;
  const int M = P * S, I = c.intermediate, heads = c.heads;
  const int Mp = (M + 127) / 128 * 128;
  const int rows_per_block = 8;                                      // warps per block of the LayerNorm kernels
  const unsigned ln_blocks = (unsigned)((M + rows_per_block - 1) / rows_per_block);             // embed LN: one row per warp
  const unsigned ln4_blocks = (unsigned)((M + rows_per_block * kLnRows - 1) / (rows_per_block * kLnRows));
  ProfScope ps(ctx, SB_PROF_CE, st, 3 + (int)m->layers.size() * 7);
  int32_t* cu = m->cu;
  const int32_t* m_dev = cu + P;  // packed row count of this pass (device side only)
  const bool cls_tail = H % 32 == 0 && H / heads == 32;   // last layer on the P [CLS] rows only
  const bool h16 = m->fp16_stream && cls_tail;            // fp16 residual stream (see CeModel::fp16_stream)
  ce_cu_kernel<<<1, 1024, 0, st>>>(lens, P, S, cu, m->stats);
  SB_CUDA(cudaGetLastError());
  ce_embed_ln_kernel<H><<<ln_blocks, rows_per_block * 32, 0, st>>>(ids, tts, lens, cu, M, S, c.vocab_size, c.type_vocab,
                                                                   m->word_emb, m->pos_emb, m->type_emb, m->emb_ln_g,
                                                                   m->emb_ln_b, c.ln_eps, h16 ? nullptr : m->x32, m->x16);
  SB_CUDA(cudaGetLastError());
  int rc;
  const int Pp = (P + 127) / 128 * 128;
  const unsigned cls_ln_blocks = (unsigned)((P + rows_per_block * kLnRows - 1) / (rows_per_block * kLnRows));
  for (size_t li = 0; li < m->layers.size(); ++li) {
    CeLayer& L = m->layers[li];
    if ((rc = ce_gemm_launch(CE_EPI_BIAS_F16, m->m_x16, L.m_wqkv, Mp, 3 * H, H, L.bqkv, nullptr, m->qkv16, nullptr, st,
                             m_dev)))
      return rc;
    if (li + 1 == m->layers.size() && cls_tail) {
      // last layer: K/V of every token, everything else for the P [CLS] rows only
      ce_attention_cls_kernel<<<(unsigned)((P * heads + 3) / 4), 128, 0, st>>>(m->qkv16, lens, cu, P, S, H, heads,
                                                                              h16 ? nullptr : m->x32, m->x16, m->ctxcls16,
                                                                              m->xcls32);
      SB_CUDA(cudaGetLastError());
      if ((rc = ce_gemm_launch(CE_EPI_BIAS_RES_F32, m->m_ctxcls16, L.m_wo, Pp, H, H, L.bo, m->xcls32, nullptr,
                               m->precls32, st)))
        return rc;
      ce_ln_kernel<H, float><<<cls_ln_blocks, rows_per_block * 32, 0, st>>>(m->precls32, P, nullptr, L.ln1_g, L.ln1_b,
                                                                            c.ln_eps, m->xcls32, m->xcls16);
      SB_CUDA(cudaGetLastError());
      if ((rc = ce_gemm_launch(CE_EPI_BIAS_GELU_F16, m->m_xcls16, L.m_w1, Pp, I, H, L.b1, nullptr, m->ffncls16, nullptr,
                               st)))
        return rc;
      if ((rc = ce_gemm_launch(CE_EPI_BIAS_RES_F32, m->m_ffncls16, L.m_w2, Pp, H, I, L.b2, m->xcls32, nullptr,
                               m->precls32, st)))
        return rc;
      ce_ln_kernel<H, float><<<cls_ln_blocks, rows_per_block * 32, 0, st>>>(m->precls32, P, nullptr, L.ln2_g, L.ln2_b,
                                                                            c.ln_eps, m->xcls32, m->xcls16);
      SB_CUDA(cudaGetLastError());
      if (cls_out) {  // embedder: hand the final [CLS] states over instead of running the classifier head
        SB_CUDA(cudaMemcpyAsync(cls_out, m->xcls32, (size_t)P * H * 4, cudaMemcpyDeviceToDevice, st));
        return SB_OK;
      }
      ce_head_kernel<<<(P + kHeadPairs - 1) / kHeadPairs, 512, (size_t)kHeadPairs * (H + 32) * sizeof(float), st>>>(
          m->xcls32, nullptr, P, H, m->pool_w, m->pool_b, m->cls_w, m->cls_b, logits, sig);
      SB_CUDA(cudaGetLastError());
      return SB_OK;
    }
    if (S <= 128 && heads % 3 == 0)
      ce_attention_mma_kernel<128, 3><<<P * (heads / 3), 128, 0, st>>>(m->qkv16, lens, cu, S, H, heads, m->ctx16);
    else if (S <= 128 && heads % 2 == 0)
      ce_attention_mma_kernel<128, 2><<<P * (heads / 2), 128, 0, st>>>(m->qkv16, lens, cu, S, H, heads, m->ctx16);
    else if (S <= 128)
      ce_attention_mma_kernel<128, 1><<<P * heads, 128, 0, st>>>(m->qkv16, lens, cu, S, H, heads, m->ctx16);
    else if (S <= 256)
      ce_attention_mma_kernel<256, 1><<<P * heads, 128, 0, st>>>(m->qkv16, lens, cu, S, H, heads, m->ctx16);
    else {
      const size_t att_smem = (size_t)2 * S * 32 * sizeof(float);
      SB_CUDA(cudaFuncSetAttribute(ce_attention_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)att_smem));
      ce_attention_kernel<32><<<P * heads, 128, att_smem, st>>>(m->qkv16, lens, cu, S, H, heads, m->ctx16);
    }
    SB_CUDA(cudaGetLastError());
    if (h16) {
      // fp16 residual stream: pre16 = fp16(ctx Wo^T + bo + x16), x16 = LN(pre16); the same for the FFN
      if ((rc = ce_gemm_launch(CE_EPI_BIAS_RES16_F16, m->m_ctx16, L.m_wo, Mp, H, H, L.bo,
                               reinterpret_cast<const float*>(m->x16), m->pre16, nullptr, st, m_dev)))
        return rc;
      ce_ln_kernel<H, __half><<<ln4_blocks, rows_per_block * 32, 0, st>>>(m->pre16, M, m_dev, L.ln1_g, L.ln1_b, c.ln_eps,
                                                                         nullptr, m->x16);
      SB_CUDA(cudaGetLastError());
      if ((rc = ce_gemm_launch(CE_EPI_BIAS_GELU_F16, m->m_x16, L.m_w1, Mp, I, H, L.b1, nullptr, m->ffn16, nullptr, st,
                               m_dev)))
        return rc;
      if ((rc = ce_gemm_launch(CE_EPI_BIAS_RES16_F16, m->m_ffn16, L.m_w2, Mp, H, I, L.b2,
                               reinterpret_cast<const float*>(m->x16), m->pre16, nullptr, st, m_dev)))
        return rc;
      ce_ln_kernel<H, __half><<<ln4_blocks, rows_per_block * 32, 0, st>>>(m->pre16, M, m_dev, L.ln2_g, L.ln2_b, c.ln_eps,
                                                                         nullptr, m->x16);
      SB_CUDA(cudaGetLastError());
      continue;
    }
    if ((rc = ce_gemm_launch(CE_EPI_BIAS_RES_F32, m->m_ctx16, L.m_wo, Mp, H, H, L.bo, m->x32, nullptr, m->pre32, st,
                             m_dev)))
      return rc;
    ce_ln_kernel<H, float><<<ln4_blocks, rows_per_block * 32, 0, st>>>(m->pre32, M, m_dev, L.ln1_g, L.ln1_b, c.ln_eps,
                                                                      m->x32, m->x16);
    SB_CUDA(cudaGetLastError());
    if ((rc = ce_gemm_launch(CE_EPI_BIAS_GELU_F16, m->m_x16, L.m_w1, Mp, I, H, L.b1, nullptr, m->ffn16, nullptr, st,
                             m_dev)))
      return rc;
    if ((rc = ce_gemm_launch(CE_EPI_BIAS_RES_F32, m->m_ffn16, L.m_w2, Mp, H, I, L.b2, m->x32, nullptr, m->pre32, st,
                             m_dev)))
      return rc;
    ce_ln_kernel<H, float><<<ln4_blocks, rows_per_block * 32, 0, st>>>(m->pre32, M, m_dev, L.ln2_g, L.ln2_b, c.ln_eps,
                                                                      m->x32, m->x16);
    SB_CUDA(cudaGetLastError());
  }
  SB_REQUIRE(cls_out == nullptr, SB_ERR_UNSUPPORTED, "encoder output needs 32-wide attention heads");
  ce_head_kernel<<<(P + kHeadPairs - 1) / kHeadPairs, 512, (size_t)kHeadPairs * (H + 32) * sizeof(float), st>>>(
      m->x32, cu, P, H, m->pool_w, m->pool_b, m->cls_w, m->cls_b, logits, sig);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

// m = the reranker (ctx->ce: logits / sigmoid out) or the embedder (ctx->enc: cls_out = final [CLS] states [P,H])
int ce_forward_dispatch(sb_ctx* ctx, CeModel* m, const int32_t* ids, const int32_t* tts, const int32_t* lens, int P,
                        int S, float* logits, float* sig, float* cls_out, cudaStream_t st) {
  SB_REQUIRE(m != nullptr, SB_ERR_STATE, "no model loaded (sb_ce_load / sb_enc_load)");
  SB_REQUIRE(S > 0 && S <= m->cfg.max_pos, SB_ERR_ARG, "sb_ce_score: sequence length %d exceeds max_pos %d", S,
             m->cfg.max_pos);
  SB_REQUIRE(S <= 512, SB_ERR_UNSUPPORTED, "sb_ce_score: sequence length %d > 512", S);
  int rc = ensure_workspace(m, P, (int64_t)P * S, st);
  if (rc) return rc;
  switch (m->cfg.hidden) {
    case 384: return ce_forward<384>(ctx, m, ids, tts, lens, P, S, logits, sig, cls_out, st);
    case 128: return ce_forward<128>(ctx, m, ids, tts, lens, P, S, logits, sig, cls_out, st);
    case 256: return ce_forward<256>(ctx, m, ids, tts, lens, P, S, logits, sig, cls_out, st);
    case 768: return ce_forward<768>(ctx, m, ids, tts, lens, P, S, logits, sig, cls_out, st);
  }
  sb_set_error("sb_ce_score: unsupported hidden size %d", m->cfg.hidden);
  return SB_ERR_UNSUPPORTED;
}

__global__ void f16_to_f32_kernel(const __half* __restrict__ in, float* __restrict__ out, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __half2float(in[i]);
}

// [CLS] query [SEP] doc [SEP] framing on the device for every (query, candidate) pair of a batch.
__global__ void ce_build_pairs_kernel(const int32_t* __restrict__ q_tok, const int32_t* __restrict__ q_len, int lq,
                                      const int64_t* __restrict__ cand_ids, const int32_t* __restrict__ cand_cnt, int k,
                                      int pair0, int n_pairs, const uint16_t* __restrict__ doc_tok,
                                      const int32_t* __restrict__ doc_len, int ld, int64_t n_docs, int64_t id_base, int S,
                                      int32_t* __restrict__ ids, int32_t* __restrict__ tts, int32_t* __restrict__ lens) {
  const int pl = blockIdx.x;  // pair index inside this chunk
  if (pl >= n_pairs) return;
  const int pair = pair0 + pl, b = pair / k, j = pair % k;
  const bool valid = j < cand_cnt[b];
  const int64_t row = valid ? cand_ids[(size_t)b * k + j] - id_base : -1;
  const int nq = min(max(q_len[b], 0), min(lq, S / 2 - 2 > 0 ? S / 2 - 2 : 1));
  int nd = (valid && row >= 0 && row < n_docs) ? min(doc_len[row], ld) : 0;
  nd = min(nd, S - nq - 3);
  if (nd < 0) nd = 0;
  const int total = valid ? nq + nd + 3 : 2;
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    int id = 0, tt = 0;
    if (valid) {
      if (s == 0) id = 101;
      else if (s <= nq) id = q_tok[(size_t)b * lq + s - 1];
      else if (s == nq + 1) id = 102;
      else if (s < nq + 2 + nd) { id = doc_tok[(size_t)row * ld + (s - nq - 2)]; tt = 1; }
      else if (s == nq + 2 + nd) { id = 102; tt = 1; }
    } else {
      if (s == 0) id = 101;
      else if (s == 1) id = 102;
    }
    ids[(size_t)pl * S + s] = id;
    tts[(size_t)pl * S + s] = tt;
  }
  if (threadIdx.x == 0) lens[pl] = total;
}

// One CTA per query: order the k candidates by relevance (desc, stable on the incoming rank) and emit the best k_out.
__global__ void ce_rank_kernel(const float* __restrict__ sig, const int64_t* __restrict__ cand_ids,
                               const int32_t* __restrict__ cand_cnt, int k, int k_out, int64_t* __restrict__ out_ids,
                               float* __restrict__ out_scores, int32_t* __restrict__ out_counts) {
  extern __shared__ float rk_sm[];
  const int b = blockIdx.x, n = min(cand_cnt[b], k);
  for (int j = threadIdx.x; j < n; j += blockDim.x) rk_sm[j] = sig[(size_t)b * k + j];
  __syncthreads();
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    const float s = rk_sm[j];
    int pos = 0;
    for (int i = 0; i < n; ++i) pos += (rk_sm[i] > s) || (rk_sm[i] == s && i < j);
    if (pos < k_out) {
      out_ids[(size_t)b * k_out + pos] = cand_ids[(size_t)b * k + j];
      out_scores[(size_t)b * k_out + pos] = s;
    }
  }
  for (int j = n + threadIdx.x; j < k_out; j += blockDim.x) {
    out_ids[(size_t)b * k_out + j] = -1;
    out_scores[(size_t)b * k_out + j] = 0.f;
  }
  if (threadIdx.x == 0) out_counts[b] = min(n, k_out);
}

}  // namespace

extern "C" {

// Test hook: run the tcgen05 GEMM of the cross-encoder on host fp32 operands (rounded to fp16 on the device).
int sb_ce_gemm_test(sb_ctx* ctx, const float* a, const float* w, const float* bias, const float* residual, int32_t M,
                    int32_t N, int32_t K, int32_t epi, float* out) {
  SB_REQUIRE(ctx && a && w && bias && out, SB_ERR_ARG, "sb_ce_gemm_test: NULL argument");
  SB_REQUIRE(M > 0 && N > 0 && K > 0 && N % 128 == 0 && K % 64 == 0, SB_ERR_ARG, "sb_ce_gemm_test: bad shape");
  SB_REQUIRE((epi != CE_EPI_BIAS_RES_F32 && epi != CE_EPI_BIAS_RES16_F16) || residual, SB_ERR_ARG,
             "sb_ce_gemm_test: residual required");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  cudaStream_t st = ctx->stream;
  const int Mp = (M + 127) / 128 * 128;
  std::vector<void*> pool;
  struct Free { std::vector<void*>& p; ~Free() { for (void* x : p) cudaFree(x); } } fr{pool};
  float *a32, *w32, *b32, *r32 = nullptr, *o32, *o32b;
  __half *a16, *w16, *o16;
  int rc;
  if ((rc = dev_alloc(pool, (void**)&a32, (size_t)Mp * K * 4))) return rc;
  if ((rc = dev_alloc(pool, (void**)&w32, (size_t)N * K * 4))) return rc;
  if ((rc = dev_alloc(pool, (void**)&b32, (size_t)N * 4))) return rc;
  if ((rc = dev_alloc(pool, (void**)&r32, (size_t)Mp * N * 4))) return rc;
  if ((rc = dev_alloc(pool, (void**)&o32, (size_t)Mp * N * 4))) return rc;
  if ((rc = dev_alloc(pool, (void**)&o32b, (size_t)Mp * N * 4))) return rc;
  if ((rc = dev_alloc(pool, (void**)&a16, (size_t)Mp * K * 2))) return rc;
  if ((rc = dev_alloc(pool, (void**)&w16, (size_t)N * K * 2))) return rc;
  if ((rc = dev_alloc(pool, (void**)&o16, (size_t)Mp * N * 2))) return rc;
  SB_CUDA(cudaMemsetAsync(a32, 0, (size_t)Mp * K * 4, st));
  SB_CUDA(cudaMemsetAsync(r32, 0, (size_t)Mp * N * 4, st));
  SB_CUDA(cudaMemcpyAsync(a32, a, (size_t)M * K * 4, cudaMemcpyHostToDevice, st));
  SB_CUDA(cudaMemcpyAsync(w32, w, (size_t)N * K * 4, cudaMemcpyHostToDevice, st));
  SB_CUDA(cudaMemcpyAsync(b32, bias, (size_t)N * 4, cudaMemcpyHostToDevice, st));
  if (residual) SB_CUDA(cudaMemcpyAsync(r32, residual, (size_t)M * N * 4, cudaMemcpyHostToDevice, st));
  f32_to_f16_kernel<<<(unsigned)(((size_t)Mp * K + 255) / 256), 256, 0, st>>>(a32, a16, (int64_t)Mp * K);
  f32_to_f16_kernel<<<(unsigned)(((size_t)N * K + 255) / 256), 256, 0, st>>>(w32, w16, (int64_t)N * K);
  CUtensorMap ma, mw;
  if ((rc = ce_make_tensor_map(&ma, a16, Mp, K))) return rc;
  if ((rc = ce_make_tensor_map(&mw, w16, N, K))) return rc;
  const float* res_arg = r32;
  if (epi == CE_EPI_BIAS_RES16_F16) {   // the fp16 residual stream: the residual operand is fp16 (rounded here)
    __half* r16 = nullptr;
    if ((rc = dev_alloc(pool, (void**)&r16, (size_t)Mp * N * 2))) return rc;
    f32_to_f16_kernel<<<(unsigned)(((size_t)Mp * N + 255) / 256), 256, 0, st>>>(r32, r16, (int64_t)Mp * N);
    res_arg = reinterpret_cast<const float*>(r16);
  }
  if ((rc = ce_gemm_launch(epi, ma, mw, Mp, N, K, b32, res_arg, o16, o32, st))) return rc;
  const float* result = o32;
  if (epi != CE_EPI_BIAS_RES_F32) {
    f16_to_f32_kernel<<<(unsigned)(((size_t)Mp * N + 255) / 256), 256, 0, st>>>(o16, o32b, (int64_t)Mp * N);
    result = o32b;
  }
  SB_CUDA(cudaGetLastError());
  SB_CUDA(cudaMemcpyAsync(out, result, (size_t)M * N * 4, cudaMemcpyDeviceToHost, st));
  SB_CUDA(cudaStreamSynchronize(st));
  return SB_OK;
}

// uploads one BERT-style model (blob layout of sentio_b200/cross_encoder.py); the caller holds ctx->mu and owns *out
static int ce_load_model(sb_ctx* ctx, const float* weights, int64_t n_floats, const sb_ce_config* cfg, CeModel** out) {
  const int V = cfg->vocab_size, H = cfg->hidden, L = cfg->layers, I = cfg->intermediate, Pm = cfg->max_pos,
            T = cfg->type_vocab;
  SB_REQUIRE(V > 0 && H > 0 && L > 0 && I > 0 && Pm > 0 && T > 0 && cfg->heads > 0, SB_ERR_ARG, "sb_ce_load: bad config");
  SB_REQUIRE(H == 128 || H == 256 || H == 384 || H == 768, SB_ERR_UNSUPPORTED,
             "sb_ce_load: hidden size %d not supported (128/256/384/768)", H);
  SB_REQUIRE(H / cfg->heads == 32 && H % cfg->heads == 0, SB_ERR_UNSUPPORTED,
             "sb_ce_load: head dimension must be 32 (hidden %d, heads %d)", H, cfg->heads);
  SB_REQUIRE(I % 128 == 0 && H % 128 == 0, SB_ERR_UNSUPPORTED, "sb_ce_load: hidden/intermediate must be multiples of 128");
  const int64_t per_layer = 4ll * H * H + 4ll * H + 2ll * H + (int64_t)I * H + I + (int64_t)H * I + H + 2ll * H;
  const int64_t expect = (int64_t)V * H + (int64_t)Pm * H + (int64_t)T * H + 2ll * H + L * per_layer + (int64_t)H * H +
                         H + H + 1;
  SB_REQUIRE(n_floats == expect, SB_ERR_ARG, "sb_ce_load: blob has %lld floats, config needs %lld", (long long)n_floats,
             (long long)expect);
  cudaStream_t st = ctx->stream;
  SB_CUDA(cudaStreamSynchronize(st));
  CeModel* m = new CeModel();
  m->cfg = *cfg;
  const float* src = weights;
  int rc = SB_OK;
#define CE_TRY(expr)            \
  if ((rc = (expr)) != SB_OK) { \
    ce_model_free(m);           \
    return rc;                  \
  }
  CE_TRY(upload_f32(m, src, &m->word_emb, (size_t)V * H, st));
  CE_TRY(upload_f32(m, src, &m->pos_emb, (size_t)Pm * H, st));
  CE_TRY(upload_f32(m, src, &m->type_emb, (size_t)T * H, st));
  CE_TRY(upload_f32(m, src, &m->emb_ln_g, H, st));
  CE_TRY(upload_f32(m, src, &m->emb_ln_b, H, st));
  m->layers.resize(L);
  for (int l = 0; l < L; ++l) {
    CeLayer& Ly = m->layers[l];
    CE_TRY(dev_alloc(m->allocs, (void**)&Ly.wqkv, (size_t)3 * H * H * 2));
    CE_TRY(dev_alloc(m->allocs, (void**)&Ly.bqkv, (size_t)3 * H * 4));
    for (int part = 0; part < 3; ++part) {  // blob order: Wq bq Wk bk Wv bv -> fused [3H,H] weight / [3H] bias
      CE_TRY(upload_f16(ctx, src, Ly.wqkv + (size_t)part * H * H, (size_t)H * H, st));
      SB_CUDA(cudaMemcpyAsync(Ly.bqkv + (size_t)part * H, src, (size_t)H * 4, cudaMemcpyHostToDevice, st));
      src += H;
    }
    CE_TRY(dev_alloc(m->allocs, (void**)&Ly.wo, (size_t)H * H * 2));
    CE_TRY(upload_f16(ctx, src, Ly.wo, (size_t)H * H, st));
    CE_TRY(upload_f32(m, src, &Ly.bo, H, st));
    CE_TRY(upload_f32(m, src, &Ly.ln1_g, H, st));
    CE_TRY(upload_f32(m, src, &Ly.ln1_b, H, st));
    CE_TRY(dev_alloc(m->allocs, (void**)&Ly.w1, (size_t)I * H * 2));
    CE_TRY(upload_f16(ctx, src, Ly.w1, (size_t)I * H, st));
    CE_TRY(upload_f32(m, src, &Ly.b1, I, st));
    CE_TRY(dev_alloc(m->allocs, (void**)&Ly.w2, (size_t)H * I * 2));
    CE_TRY(upload_f16(ctx, src, Ly.w2, (size_t)H * I, st));
    CE_TRY(upload_f32(m, src, &Ly.b2, H, st));
    CE_TRY(upload_f32(m, src, &Ly.ln2_g, H, st));
    CE_TRY(upload_f32(m, src, &Ly.ln2_b, H, st));
    CE_TRY(ce_make_tensor_map(&Ly.m_wqkv, Ly.wqkv, 3 * H, H));
    CE_TRY(ce_make_tensor_map(&Ly.m_wo, Ly.wo, H, H));
    CE_TRY(ce_make_tensor_map(&Ly.m_w1, Ly.w1, I, H));
    CE_TRY(ce_make_tensor_map(&Ly.m_w2, Ly.w2, H, I));
  }
  CE_TRY(upload_f32(m, src, &m->pool_w, (size_t)H * H, st));
  CE_TRY(upload_f32(m, src, &m->pool_b, H, st));
  CE_TRY(upload_f32(m, src, &m->cls_w, H, st));
  CE_TRY(upload_f32(m, src, &m->cls_b, 1, st));
#undef CE_TRY
  SB_CUDA(cudaStreamSynchronize(st));
  *out = m;
  return SB_OK;
}

}  // extern "C"

namespace {

// out[p, :] = (normalize) ( W_proj x_cls[p] + b_proj )   (W_proj == NULL: identity on the H-dim [CLS] state).
// One CTA per kHeadPairs inputs, a warp per output column: every projection row is read once per CTA.
__global__ void __launch_bounds__(256) enc_project_kernel(const float* __restrict__ cls, int P, int H,
                                                          const float* __restrict__ pw, const float* __restrict__ pb,
                                                          int D, int normalize, float* __restrict__ out) {
  extern __shared__ float ep_sm[];   // x[kHeadPairs][H], y[kHeadPairs][D], norm[kHeadPairs]
  float* x = ep_sm;
  float* y = ep_sm + kHeadPairs * H;
  float* nrm = y + (size_t)kHeadPairs * D;
  const int p0 = blockIdx.x * kHeadPairs, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int np = min(kHeadPairs, P - p0);
  for (int i = threadIdx.x; i < kHeadPairs * H; i += blockDim.x) x[i] = (i / H) < np ? cls[(size_t)p0 * H + i] : 0.f;
  __syncthreads();
  for (int o = warp; o < D; o += nw) {
    float acc[kHeadPairs];
#pragma unroll
    for (int q = 0; q < kHeadPairs; ++q) acc[q] = 0.f;
    if (pw) {
      for (int c = lane; c < H; c += 32) {
        const float wv = pw[(size_t)o * H + c];
#pragma unroll
        for (int q = 0; q < kHeadPairs; ++q) acc[q] = fmaf(wv, x[q * H + c], acc[q]);
      }
#pragma unroll
      for (int q = 0; q < kHeadPairs; ++q)
        for (int s = 16; s; s >>= 1) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], s);
    }
    if (lane == 0)
#pragma unroll
      for (int q = 0; q < kHeadPairs; ++q) y[(size_t)q * D + o] = pw ? acc[q] + pb[o] : x[q * H + o];
  }
  __syncthreads();
  if (warp < kHeadPairs) {  // L2 norm of row `warp`
    float ss = 0.f;
    for (int o = lane; o < D; o += 32) ss = fmaf(y[(size_t)warp * D + o], y[(size_t)warp * D + o], ss);
    for (int s = 16; s; s >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, s);
    if (lane == 0) nrm[warp] = (normalize && ss > 0.f) ? rsqrtf(ss) : 1.f;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < np * D; i += blockDim.x) out[(size_t)p0 * D + i] = y[i] * nrm[i / D];
}

int enc_embed_enqueue(sb_ctx* ctx, const int32_t* ids, const int32_t* tts, const int32_t* lens, int P, int S, int normalize,
                      float* out_dev, cudaStream_t st) {
  CeModel* m = ctx->enc;
  SB_REQUIRE(m != nullptr, SB_ERR_STATE, "sb_enc_embed: no encoder loaded (sb_enc_load)");
  const int H = m->cfg.hidden, D = m->proj_w ? m->out_dim : H;
  int rc = ctx->misc3_dev.reserve((size_t)P * H * 4 + 64);
  if (rc) return rc;
  float* cls = ctx->misc3_dev.as<float>();
  if ((rc = ce_forward_dispatch(ctx, m, ids, tts, lens, P, S, nullptr, nullptr, cls, st))) return rc;
  const size_t smem = ((size_t)kHeadPairs * (H + D) + kHeadPairs + 8) * sizeof(float);
  SB_REQUIRE(smem <= ctx->smem_optin, SB_ERR_UNSUPPORTED, "sb_enc_embed: output dimension %d too large", D);
  SB_CUDA(cudaFuncSetAttribute(enc_project_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ctx->launches += 1;
  enc_project_kernel<<<(P + kHeadPairs - 1) / kHeadPairs, 256, smem, st>>>(cls, P, H, m->proj_w, m->proj_b, D, normalize,
                                                                          out_dev);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

}  // namespace

extern "C" {

int sb_ce_load(sb_ctx* ctx, const float* weights, int64_t n_floats, const sb_ce_config* cfg) {
  SB_REQUIRE(ctx && weights && cfg, SB_ERR_ARG, "sb_ce_load: NULL argument");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  CeModel* m = nullptr;
  int rc = ce_load_model(ctx, weights, n_floats, cfg, &m);
  if (rc) return rc;
  if (ctx->ce) ce_model_free(ctx->ce);
  m->fp16_stream = true;   // the reranker runs on the fp16 residual stream (see CeModel::fp16_stream)
  ctx->ce = m;
  return SB_OK;
}

int sb_enc_load(sb_ctx* ctx, const float* weights, int64_t n_floats, const sb_ce_config* cfg, const float* proj_w,
                const float* proj_b, int32_t out_dim) {
  SB_REQUIRE(ctx && weights && cfg, SB_ERR_ARG, "sb_enc_load: NULL argument");
  SB_REQUIRE((proj_w == nullptr) == (proj_b == nullptr) && (proj_w == nullptr || out_dim > 0), SB_ERR_ARG,
             "sb_enc_load: proj_w / proj_b / out_dim must be given together");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  CeModel* m = nullptr;
  int rc = ce_load_model(ctx, weights, n_floats, cfg, &m);
  if (rc) return rc;
  if (proj_w) {
    const float* src = proj_w;
    if ((rc = upload_f32(m, src, &m->proj_w, (size_t)out_dim * cfg->hidden, ctx->stream)) == SB_OK) {
      src = proj_b;
      rc = upload_f32(m, src, &m->proj_b, (size_t)out_dim, ctx->stream);
    }
    if (rc) {
      ce_model_free(m);
      return rc;
    }
    m->out_dim = out_dim;
    SB_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  if (ctx->enc) ce_model_free(ctx->enc);
  ctx->enc = m;
  return SB_OK;
}

int32_t sb_enc_dim(sb_ctx* ctx) {
  if (!ctx || !ctx->enc) return -1;
  return ctx->enc->proj_w ? ctx->enc->out_dim : ctx->enc->cfg.hidden;
}

int sb_enc_embed_dev(sb_ctx* ctx, const int32_t* input_ids_dev, const int32_t* token_type_dev, const int32_t* lengths_dev,
                     int32_t P, int32_t S, int32_t normalize, float* out_dev, void* stream) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_enc_embed_dev: ctx is NULL");
  SB_REQUIRE(P >= 0 && S > 0, SB_ERR_ARG, "sb_enc_embed_dev: bad P=%d S=%d", P, S);
  if (P == 0) return SB_OK;
  SB_REQUIRE(input_ids_dev && token_type_dev && lengths_dev && out_dev, SB_ERR_ARG, "sb_enc_embed_dev: NULL buffer");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  return enc_embed_enqueue(ctx, input_ids_dev, token_type_dev, lengths_dev, P, S, normalize, out_dev,
                           pick_stream(ctx, stream));
}

int sb_enc_embed(sb_ctx* ctx, const int32_t* input_ids, const int32_t* token_type, const int32_t* lengths, int32_t P,
                 int32_t S, int32_t normalize, float* out) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_enc_embed: ctx is NULL");
  SB_REQUIRE(P >= 0 && S > 0, SB_ERR_ARG, "sb_enc_embed: bad P=%d S=%d", P, S);
  if (P == 0) return SB_OK;
  SB_REQUIRE(input_ids && token_type && lengths && out, SB_ERR_ARG, "sb_enc_embed: NULL buffer");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  SB_REQUIRE(ctx->enc != nullptr, SB_ERR_STATE, "sb_enc_embed: no encoder loaded (sb_enc_load)");
  cudaStream_t st = ctx->stream;
  const int D = ctx->enc->proj_w ? ctx->enc->out_dim : ctx->enc->cfg.hidden;
  const size_t nb = (size_t)P * S * 4;
  int rc;
  if ((rc = ctx->pin_in.reserve(2 * nb + (size_t)P * 4))) return rc;
  if ((rc = ctx->q_dev.reserve(2 * nb + (size_t)P * 4))) return rc;
  uint8_t* pi = ctx->pin_in.as<uint8_t>();
  memcpy(pi, input_ids, nb);
  memcpy(pi + nb, token_type, nb);
  memcpy(pi + 2 * nb, lengths, (size_t)P * 4);
  SB_CUDA(cudaMemcpyAsync(ctx->q_dev.p, pi, 2 * nb + (size_t)P * 4, cudaMemcpyHostToDevice, st));
  uint8_t* dv = ctx->q_dev.as<uint8_t>();
  if ((rc = ctx->out_sc_dev.reserve((size_t)P * D * 4))) return rc;
  if ((rc = enc_embed_enqueue(ctx, (const int32_t*)dv, (const int32_t*)(dv + nb), (const int32_t*)(dv + 2 * nb), P, S,
                              normalize, ctx->out_sc_dev.as<float>(), st)))
    return rc;
  if ((rc = ctx->pin_out.reserve((size_t)P * D * 4))) return rc;
  SB_CUDA(cudaMemcpyAsync(ctx->pin_out.p, ctx->out_sc_dev.p, (size_t)P * D * 4, cudaMemcpyDeviceToHost, st));
  SB_CUDA(cudaStreamSynchronize(st));
  memcpy(out, ctx->pin_out.p, (size_t)P * D * 4);
  return SB_OK;
}


int sb_ce_score_dev(sb_ctx* ctx, const int32_t* input_ids_dev, const int32_t* token_type_dev, const int32_t* lengths_dev,
                    int32_t P, int32_t S, float* out_logits_dev, float* out_sigmoid_dev, void* stream) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_ce_score_dev: ctx is NULL");
  SB_REQUIRE(P >= 0 && S > 0, SB_ERR_ARG, "sb_ce_score_dev: bad P=%d S=%d", P, S);
  if (P == 0) return SB_OK;
  SB_REQUIRE(input_ids_dev && token_type_dev && lengths_dev && out_logits_dev && out_sigmoid_dev, SB_ERR_ARG,
             "sb_ce_score_dev: NULL buffer");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  return ce_forward_dispatch(ctx, ctx->ce, input_ids_dev, token_type_dev, lengths_dev, P, S, out_logits_dev,
                             out_sigmoid_dev, nullptr, pick_stream(ctx, stream));
}

int sb_ce_stats(sb_ctx* ctx, int64_t* out3, int32_t reset) {
  SB_REQUIRE(ctx != nullptr && out3 != nullptr, SB_ERR_ARG, "sb_ce_stats: NULL argument");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  out3[0] = out3[1] = out3[2] = 0;
  if (!ctx->ce || !ctx->ce->stats) return SB_OK;
  SB_CUDA(cudaDeviceSynchronize());
  unsigned long long h[3];
  SB_CUDA(cudaMemcpy(h, ctx->ce->stats, sizeof(h), cudaMemcpyDeviceToHost));
  for (int i = 0; i < 3; ++i) out3[i] = (int64_t)h[i];
  if (reset) SB_CUDA(cudaMemset(ctx->ce->stats, 0, sizeof(h)));
  return SB_OK;
}

int sb_ce_score(sb_ctx* ctx, const int32_t* input_ids, const int32_t* token_type, const int32_t* lengths, int32_t P,
                int32_t S, float* out_logits, float* out_sigmoid) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_ce_score: ctx is NULL");
  SB_REQUIRE(P >= 0 && S > 0, SB_ERR_ARG, "sb_ce_score: bad P=%d S=%d", P, S);
  if (P == 0) return SB_OK;
  SB_REQUIRE(input_ids && token_type && lengths && out_logits && out_sigmoid, SB_ERR_ARG, "sb_ce_score: NULL buffer");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  cudaStream_t st = ctx->stream;
  const size_t nb = (size_t)P * S * 4;
  int rc;
  if ((rc = ctx->pin_in.reserve(2 * nb + (size_t)P * 4))) return rc;
  if ((rc = ctx->q_dev.reserve(2 * nb + (size_t)P * 4))) return rc;
  uint8_t* pi = ctx->pin_in.as<uint8_t>();
  memcpy(pi, input_ids, nb);
  memcpy(pi + nb, token_type, nb);
  memcpy(pi + 2 * nb, lengths, (size_t)P * 4);
  SB_CUDA(cudaMemcpyAsync(ctx->q_dev.p, pi, 2 * nb + (size_t)P * 4, cudaMemcpyHostToDevice, st));
  uint8_t* dv = ctx->q_dev.as<uint8_t>();
  if ((rc = ctx->out_sc_dev.reserve((size_t)P * 8))) return rc;
  float* dl = ctx->out_sc_dev.as<float>();
  float* ds = dl + P;
  if ((rc = ce_forward_dispatch(ctx, ctx->ce, (const int32_t*)dv, (const int32_t*)(dv + nb),
                                (const int32_t*)(dv + 2 * nb), P, S, dl, ds, nullptr, st)))
    return rc;
  if ((rc = ctx->pin_out.reserve((size_t)P * 8))) return rc;
  SB_CUDA(cudaMemcpyAsync(ctx->pin_out.p, dl, (size_t)P * 8, cudaMemcpyDeviceToHost, st));
  SB_CUDA(cudaStreamSynchronize(st));
  memcpy(out_logits, ctx->pin_out.p, (size_t)P * 4);
  memcpy(out_sigmoid, ctx->pin_out.as<uint8_t>() + (size_t)P * 4, (size_t)P * 4);
  return SB_OK;
}


int sb_ce_tokens_load(sb_ctx* ctx, const uint16_t* doc_tok, const int32_t* doc_len, int64_t n_docs, int32_t ld,
                      int64_t id_base) {
  SB_REQUIRE(ctx && (n_docs == 0 || (doc_tok && doc_len)) && n_docs >= 0 && ld > 0, SB_ERR_ARG,
             "sb_ce_tokens_load: bad arguments");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  SB_CUDA(cudaStreamSynchronize(ctx->stream));
  CeDocTokens*& dt = ctx->ce_tokens;
  if (dt) {
    if (dt->tok) cudaFree(dt->tok);
    if (dt->len) cudaFree(dt->len);
    delete dt;
    dt = nullptr;
  }
  dt = new CeDocTokens();
  dt->n = n_docs;
  dt->ld = ld;
  dt->id_base = id_base;
  if (n_docs) {
    SB_CUDA(cudaMalloc(&dt->tok, (size_t)n_docs * ld * 2));
    SB_CUDA(cudaMalloc(&dt->len, (size_t)n_docs * 4));
    SB_CUDA(cudaMemcpy(dt->tok, doc_tok, (size_t)n_docs * ld * 2, cudaMemcpyHostToDevice));
    SB_CUDA(cudaMemcpy(dt->len, doc_len, (size_t)n_docs * 4, cudaMemcpyHostToDevice));
  }
  return SB_OK;
}

int sb_rerank_dev(sb_ctx* ctx, const int32_t* q_tok_dev, const int32_t* q_len_dev, int32_t lq,
                  const int64_t* cand_ids_dev, const int32_t* cand_cnt_dev, int32_t B, int32_t k, int32_t S,
                  int32_t k_out, int64_t* out_ids_dev, float* out_scores_dev, int32_t* out_counts_dev, void* stream) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_rerank_dev: ctx is NULL");
  SB_REQUIRE(B >= 0 && k > 0 && k_out > 0 && lq > 0 && S >= 8, SB_ERR_ARG, "sb_rerank_dev: bad sizes");
  if (B == 0) return SB_OK;
  SB_REQUIRE(q_tok_dev && q_len_dev && cand_ids_dev && cand_cnt_dev && out_ids_dev && out_scores_dev && out_counts_dev,
             SB_ERR_ARG, "sb_rerank_dev: NULL buffer");
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  SB_REQUIRE(ctx->ce != nullptr, SB_ERR_STATE, "sb_rerank_dev: no cross-encoder loaded (sb_ce_load)");
  SB_REQUIRE(ctx->ce_tokens != nullptr && ctx->ce_tokens->n > 0, SB_ERR_STATE,
             "sb_rerank_dev: no document tokens loaded (sb_ce_tokens_load)");
  cudaStream_t st = pick_stream(ctx, stream);
  const CeDocTokens& dt = *ctx->ce_tokens;
  const int total = B * k;
  const int chunk = 2048;  // pairs per forward pass: bounds the activation workspace (~2.6 GB at S = 128)
  int rc;
  const size_t per_pair = (size_t)S * 8 + 4;
  if ((rc = ctx->misc_dev.reserve((size_t)std::min(total, chunk) * per_pair + 64))) return rc;
  if ((rc = ctx->out_sc_dev.reserve((size_t)total * 8))) return rc;
  int32_t* ids = ctx->misc_dev.as<int32_t>();
  int32_t* tts = ids + (size_t)std::min(total, chunk) * S;
  int32_t* lens = tts + (size_t)std::min(total, chunk) * S;
  float* logits = ctx->out_sc_dev.as<float>();
  float* sig = logits + total;
  for (int p0 = 0; p0 < total; p0 += chunk) {
    const int np = std::min(chunk, total - p0);
    ctx->launches += 1;
    ce_build_pairs_kernel<<<np, 128, 0, st>>>(q_tok_dev, q_len_dev, lq, cand_ids_dev, cand_cnt_dev, k, p0, np, dt.tok,
                                              dt.len, dt.ld, dt.n, dt.id_base, S, ids, tts, lens);
    SB_CUDA(cudaGetLastError());
    if ((rc = ce_forward_dispatch(ctx, ctx->ce, ids, tts, lens, np, S, logits + p0, sig + p0, nullptr, st))) return rc;
  }
  ctx->launches += 1;
  ce_rank_kernel<<<B, 128, (size_t)k * 4, st>>>(sig, cand_ids_dev, cand_cnt_dev, k, k_out, out_ids_dev, out_scores_dev,
                                               out_counts_dev);
  SB_CUDA(cudaGetLastError());
  return SB_OK;
}

}  // extern "C"
