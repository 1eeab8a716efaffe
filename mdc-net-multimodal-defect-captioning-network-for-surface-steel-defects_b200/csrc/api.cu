// api.cu -- context, error text, model handle.
#include "common.cuh"
#include <stdlib.h>
#include <string.h>

static thread_local char g_err[1024] = "";

void mdc_set_error(const char* fmt, ...) {
  va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}

extern "C" int mdc_abi_version(void) { return MDC_ABI_VERSION; }
extern "C" const char* mdc_last_error(void) { return g_err; }

extern "C" int mdc_ctx_create(int device, mdc_ctx** out) {
  MDC_CHECK_ARG(out != nullptr);
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    MDC_FAIL(-1, "mdc_ctx_create: no CUDA device (%s); this library has no CPU fallback", cudaGetErrorString(e));
  MDC_CHECK_ARG(device >= 0 && device < n);
  cudaDeviceProp p; MDC_CUDA(cudaGetDeviceProperties(&p, device));
  if (p.major != 10)
    MDC_FAIL(-1, "mdc_ctx_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, p.major, p.minor);
  mdc_ctx* c = (mdc_ctx*)calloc(1, sizeof(mdc_ctx));
  c->device = device; c->sm_count = p.multiProcessorCount;
#ifdef MDC_DEVTOOLS   // developer build only: kernel A/B switches (the product library has one path per operation)
  const char* gb = getenv("MDC_GEMM_BACKEND");
  c->gemm_backend_simt = (gb && !strcmp(gb, "simt"));
  const char* ab = getenv("MDC_ATTN_BACKEND");
  c->attn_backend_simt = (ab && !strcmp(ab, "simt"));
#endif
  *out = c; return 0;
}

extern "C" int mdc_ctx_destroy(mdc_ctx* ctx) {
  if (!ctx) return 0;
  gemm_tc_ctx_destroy(ctx);
  decode_cluster_ctx_destroy(ctx);
  free(ctx); return 0;
}

extern "C" int64_t mdc_ctx_launch_count(const mdc_ctx* ctx) { return ctx ? ctx->launches : -1; }

extern "C" int mdc_model_num_weights(const mdc_dims* d) {
  if (!d) return -1;
  return MDC_ENC_GLOBAL_SLOTS + d->enc_depth * MDC_ENC_BLOCK_SLOTS + MDC_DEC_GLOBAL_SLOTS + d->dec_layers * MDC_DEC_LAYER_SLOTS;
}

extern "C" int mdc_model_create(mdc_ctx* ctx, const mdc_dims* d, const void* const* weights, int n_weights, mdc_model** out) {
  MDC_CHECK_ARG(ctx && d && weights && out);
  MDC_CHECK_ARG(d->precision == MDC_F32 || d->precision == MDC_BF16);
  MDC_CHECK_ARG(n_weights == mdc_model_num_weights(d));
  MDC_CHECK_ARG(d->enc_dim % d->enc_heads == 0 && d->dim % d->dec_heads == 0);
  MDC_CHECK_ARG(d->enc_dim % 8 == 0 && d->dim % 32 == 0 && d->dec_ffn % 8 == 0);
  MDC_CHECK_ARG((d->dim / d->dec_heads) % 8 == 0 && (d->dim / d->dec_heads) <= 128);
  if (d->dec_layers > 0) {
    const int hd = d->dim / d->dec_heads;
    if (hd != 32 && hd != 64 && hd != 128)
      MDC_FAIL(-2, "mdc_model_create: decoder head width %d (dim %d / %d heads) is not supported: the decode kernels cover 32, 64 and 128",
               hd, d->dim, d->dec_heads);
    if (d->dim > MDC_MAX_DEC_DIM)
      MDC_FAIL(-2, "mdc_model_create: decoder dim %d is not supported: the decode kernels cover at most %d", d->dim, MDC_MAX_DEC_DIM);
  }
  MDC_CHECK_ARG(d->enc_depth == 0 || d->n_patches == (d->img_size / d->patch) * (d->img_size / d->patch));
  MDC_CHECK_ARG(d->page_tokens > 0 && d->vocab > 0 && d->vocab <= 4096 && d->max_pos > 0);
  mdc_model* m = (mdc_model*)calloc(1, sizeof(mdc_model));
  m->ctx = ctx; m->d = *d; m->n_w = n_weights;
  m->w = (const void**)malloc(sizeof(void*) * n_weights);
  memcpy(m->w, weights, sizeof(void*) * n_weights);
  *out = m; return 0;
}

extern "C" int mdc_model_destroy(mdc_model* m) {
  if (!m) return 0;
  decode_cluster_model_destroy(m);
  free(m->w); free(m); return 0;
}
