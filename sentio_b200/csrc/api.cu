// api.cu -- context lifetime + error plumbing of libsentio_b200.
#include <stdarg.h>

#include "common.cuh"

static thread_local char g_err[1024] = "";

void sb_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

void ce_model_free(CeModel* m);        // cross_encoder.cu
void ce_tokens_free(CeDocTokens* t);   // cross_encoder.cu
void bm25_build_free(Bm25Build* b);    // bm25_build.cu

extern "C" {

const char* sb_last_error(void) { return g_err; }

int sb_version(void) { return 1000; }

int sb_create(int device, sb_ctx** out) {
  SB_REQUIRE(out != nullptr, SB_ERR_ARG, "sb_create: out is NULL");
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    sb_set_error("sb_create: no CUDA device visible (%s); libsentio_b200 has no CPU fallback",
                 e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return SB_ERR_CUDA;
  }
  SB_REQUIRE(device >= 0 && device < ndev, SB_ERR_ARG, "sb_create: device %d out of range [0,%d)", device, ndev);
  DeviceGuard g(device);
  cudaDeviceProp prop;
  SB_CUDA(cudaGetDeviceProperties(&prop, device));
  SB_REQUIRE(prop.major == 10, SB_ERR_UNSUPPORTED,
             "sb_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major,
             prop.minor);
  sb_ctx* ctx = new sb_ctx();
  ctx->device = device;
  ctx->num_sms = prop.multiProcessorCount;
  ctx->smem_optin = prop.sharedMemPerBlockOptin;
  cudaError_t se = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if (se != cudaSuccess) {
    sb_set_error("sb_create: cudaStreamCreate failed: %s", cudaGetErrorString(se));
    delete ctx;
    return SB_ERR_CUDA;
  }
  *out = ctx;
  return SB_OK;
}

void sb_destroy(sb_ctx* ctx) {
  if (!ctx) return;
  DeviceGuard g(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (int s = 0; s < SB_MAX_DENSE_SLOTS; ++s) {
    if (ctx->dense[s].rows) cudaFree(ctx->dense[s].rows);
    if (ctx->dense[s].inv_norm) cudaFree(ctx->dense[s].inv_norm);
  }
  Bm25Index& b = ctx->bm25;
  if (b.indptr) cudaFree(b.indptr);
  if (b.post_doc) cudaFree(b.post_doc);
  if (b.post_ratio) cudaFree(b.post_ratio);
  if (b.dnorm) cudaFree(b.dnorm);
  if (b.idf) cudaFree(b.idf);
  if (b.dense_of_term) cudaFree(b.dense_of_term);
  if (b.dense_ratio) cudaFree(b.dense_ratio);
  if (ctx->ce) ce_model_free(ctx->ce);
  if (ctx->enc) ce_model_free(ctx->enc);
  if (ctx->ce_tokens) ce_tokens_free(ctx->ce_tokens);
  if (ctx->bm25_build) bm25_build_free(ctx->bm25_build);
  ctx->q_dev.release();
  ctx->cand_dev.release();
  ctx->out_ids_dev.release();
  ctx->out_sc_dev.release();
  ctx->out_cnt_dev.release();
  ctx->misc_dev.release();
  ctx->misc2_dev.release();
  ctx->misc3_dev.release();
  ctx->acc_dev.release();
  ctx->qn_dev.release();
  ctx->qaux_dev.release();
  ctx->doc_chars_dev.release();
  ctx->pin_in.release();
  ctx->pin_out.release();
  ctx->hyb_pin.release();
  ctx->hyb_dev.release();
  for (auto& r : ctx->prof_recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  for (auto e : ctx->prof_pool) cudaEventDestroy(e);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

void* sb_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (bytes == 0) bytes = 16;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) {
    (void)cudaGetLastError();
    sb_set_error("sb_host_alloc: cudaMallocHost(%zu) failed", bytes);
    return nullptr;
  }
  return p;
}

void sb_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

int sb_num_sms(sb_ctx* ctx) { return ctx ? ctx->num_sms : 0; }

int sb_sync(sb_ctx* ctx) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_sync: ctx is NULL");
  DeviceGuard g(ctx->device);
  SB_CUDA(cudaStreamSynchronize(ctx->stream));
  return SB_OK;
}

void* sb_stream(sb_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int64_t sb_launch_count(sb_ctx* ctx) { return ctx ? (int64_t)ctx->launches : -1; }

int sb_profile(sb_ctx* ctx, int enable) {
  SB_REQUIRE(ctx != nullptr, SB_ERR_ARG, "sb_profile: ctx is NULL");
  std::lock_guard<std::mutex> lk(ctx->mu);
  ctx->prof_on = enable != 0;
  return SB_OK;
}

int sb_profile_read(sb_ctx* ctx, int kernel_id, int64_t* n_out, double* ms_out) {
  SB_REQUIRE(ctx != nullptr && n_out && ms_out, SB_ERR_ARG, "sb_profile_read: NULL argument");
  SB_REQUIRE(kernel_id >= 0 && kernel_id < SB_PROF_COUNT, SB_ERR_ARG, "sb_profile_read: bad kernel id %d", kernel_id);
  std::lock_guard<std::mutex> lk(ctx->mu);
  DeviceGuard g(ctx->device);
  int64_t n = 0;
  double ms = 0.0;
  std::vector<sb_ctx::ProfRec> keep;
  for (auto& r : ctx->prof_recs) {
    if (r.id != kernel_id) {
      keep.push_back(r);
      continue;
    }
    SB_CUDA(cudaEventSynchronize(r.b));
    float t = 0.f;
    SB_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
    ms += t;
    ++n;
    ctx->prof_pool.push_back(r.a);
    ctx->prof_pool.push_back(r.b);
  }
  ctx->prof_recs.swap(keep);
  *n_out = n;
  *ms_out = ms;
  return SB_OK;
}

}  // extern "C"
