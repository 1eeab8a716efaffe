// common.cuh -- shared helpers for the sm_100a MDC-Net kernels.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <math.h>
#include "../../include/mdc_b200.h"
#include "ptx.cuh"

typedef __nv_bfloat16 bf16;

constexpr float LOG2E = 1.4426950408889634f;

// widest decoder model row the decode kernels build (LayerNorm-on-load / embedding operands); mdc_model_create rejects wider decoders
constexpr int MDC_MAX_DEC_DIM = 1024;

// ---- error plumbing ------------------------------------------------------------------------
void mdc_set_error(const char* fmt, ...);
#define MDC_FAIL(code, ...) do { mdc_set_error(__VA_ARGS__); return (code); } while (0)
#define MDC_CHECK_ARG(cond) do { if (!(cond)) MDC_FAIL(-2, "%s:%d: bad argument: %s", __FILE__, __LINE__, #cond); } while (0)
#define MDC_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) \
    MDC_FAIL(-3, "%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); } while (0)
#define MDC_LAUNCH_CHECK(ctx) do { cudaError_t e__ = cudaGetLastError(); if (e__ != cudaSuccess) \
    MDC_FAIL(-4, "%s:%d: kernel launch failed: %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
    if (ctx) (ctx)->launches++; } while (0)
#define MDC_TRY(call) do { int r__ = (call); if (r__ != 0) return r__; } while (0)

struct TmapCacheEntry;   // gemm_tcgen05.cu

struct mdc_ctx {
  int device;
  int sm_count;
  int64_t launches;
  int gemm_backend_simt;      // developer builds (-DMDC_DEVTOOLS) only: MDC_GEMM_BACKEND=simt forces the FFMA kernel for bf16 too
  int attn_backend_simt;
  void* tmap_cache;           // opaque, owned by gemm_tcgen05.cu
  void* encode_fn;            // cuTensorMapEncodeTiled entry point
  void* decode_state;         // opaque, owned by decode_cluster.cu (per-device occupancy / smem opt-in state)
};

#define MDC_MAX_DEVICES 32
// every entry point runs on the device its context was created for (cudaFuncSetAttribute, streams and tensor maps are per device)
#define MDC_CHECK_DEVICE(ctx) do { int dev__ = -1; MDC_CUDA(cudaGetDevice(&dev__)); if (dev__ != (ctx)->device) \
    MDC_FAIL(-5, "%s:%d: current CUDA device %d is not the context's device %d (wrap the call in a device guard)", __FILE__, __LINE__, dev__, (ctx)->device); } while (0)

struct mdc_model {
  mdc_ctx* ctx;
  mdc_dims d;
  const void** w;     // weight table copy (host array of device pointers)
  int n_w;
  void* fused_cache;  // opaque, owned by decode_cluster.cu (cached kernel parameters)
  const void* dec_pack;  // decode-loop weights packed for the fused kernel (mdc_decode_pack), caller-owned
};

// ---- typed load/store ----------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<bf16>(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }

// IEEE half operands and outputs (DESIGN 3.7): clamped to the finite range, then rounded to nearest.  fp16 has 11 significant bits, 8x
// finer than bf16: tools/error_budget_cpu.py "activations fp16" moves the logit error by < 3e-4, where bf16 activations would cost 1.4e-2
__device__ __forceinline__ float clamp_f16_range(float v) { return fminf(fmaxf(v, -65504.f), 65504.f); }
__device__ __forceinline__ __half f16_sat(float v) { return __float2half_rn(clamp_f16_range(v)); }
__device__ __forceinline__ uint32_t pack_f16x2_sat(float a, float b) { return pack_f16x2(clamp_f16_range(a), clamp_f16_range(b)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

// 8 consecutive elements -> 8 floats (128-bit load for bf16, 2x128-bit for f32); p must be 16B aligned
__device__ __forceinline__ void load8(const float* p, float* v) {
  float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void load8(const bf16* p, float* v) {
  uint4 r = *reinterpret_cast<const uint4*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) { float2 f = __bfloat1622float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
__device__ __forceinline__ void load8(const __half* p, float* v) {
  uint4 r = *reinterpret_cast<const uint4*>(p);
  const __half2* h = reinterpret_cast<const __half2*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) { float2 f = __half22float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
__device__ __forceinline__ void store8(float* p, const float* v) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void store8(bf16* p, const float* v) {
  uint4 r; __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
  *reinterpret_cast<uint4*>(p) = r;
}

// raise a kernel's dynamic-smem limit only when a launch needs more than any launch before it (one driver call, not one per launch)
// (the attribute is per device: the high-water mark is kept per device index)
#define MDC_ENSURE_SMEM(kernel, bytes)                                                                          \
  do {                                                                                                          \
    static int cur__[MDC_MAX_DEVICES];                                                                          \
    int dev__ = 0; MDC_CUDA(cudaGetDevice(&dev__));                                                             \
    if (dev__ < 0 || dev__ >= MDC_MAX_DEVICES) MDC_FAIL(-2, "device index %d out of range", dev__);             \
    if ((int)(bytes) > 48 * 1024 && (int)(bytes) > cur__[dev__]) {                                              \
      MDC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes)));        \
      cur__[dev__] = (int)(bytes);                                                                              \
    }                                                                                                           \
  } while (0)

// Paged self-attention KV pool (mdc_decode_state.kv_pool): [page][layer][head][k|v][page_tokens][hd] -- the K and V rows of one (page,
// layer, head) are one contiguous 2 * page_tokens * hd block (the fused decode kernel fetches it with ONE bulk copy).  When a row is 64
// bytes (hd = 32, 16-bit cache) the 16-byte chunk c of token r is stored at chunk c ^ ((r >> 1) & 3): the bank-conflict-free pattern of
// the fused kernel's ldmatrix reads (what TMA SWIZZLE_64B would produce).  Every writer and reader of the pool uses this layout.
template <typename TKV, int HD>
__device__ __forceinline__ int kv_chunk(int r, int c) { return (HD * (int)sizeof(TKV) == 64) ? (c ^ ((r >> 1) & 3)) : c; }

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline size_t esize(int dtype) { return dtype == MDC_BF16 ? 2 : 4; }

// ---- internal entry points shared between translation units --------------------------------
int gemm_simt_launch(mdc_ctx* ctx, int dtype, int epilogue, const void* A, int64_t lda, const void* W, int64_t ldw,
                     void* D, int64_t ldd, const float* bias, const float* aux0, int period, int M, int N, int K,
                     cudaStream_t s);
int gemm_tc_launch(mdc_ctx* ctx, int epilogue, const void* A, int64_t lda, const void* W, int64_t ldw,
                   void* D, int64_t ldd, const float* bias, const float* aux0, int period, int M, int N, int K,
                   cudaStream_t s, int f16 = 0);
int gemm_tc_supported(int M, int N, int K, int64_t lda, int64_t ldw);
void gemm_tc_ctx_destroy(mdc_ctx* ctx);
int mdc_make_tmap_2d(mdc_ctx* ctx, const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows, int swizzle_mode, void* out_map);
void decode_cluster_model_destroy(mdc_model* m);
void decode_cluster_ctx_destroy(mdc_ctx* ctx);
size_t decode_cluster_pack_bytes(const mdc_model* m);
int decode_cluster_pack(mdc_model* m, void* out, cudaStream_t s);
size_t decode_cluster_ckv_pack_bytes(const mdc_model* m, int B);
int decode_cluster_ckv_pack(mdc_model* m, const void* ckv_plain, int B, void* out, cudaStream_t s);
