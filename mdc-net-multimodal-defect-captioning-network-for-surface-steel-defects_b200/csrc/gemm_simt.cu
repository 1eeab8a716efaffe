// gemm_simt.cu -- FFMA GEMM, D = epi(A[M,K] . W[N,K]^T): the fp32 token-exact path (north_star:
// "greedy-decoded token IDs must match exactly on an fp32 path"), also usable on bf16 operands as a
// bisecting aid for the tcgen05 kernel.  Each output element is accumulated by ONE thread in
// ascending-k order with fp32 FMAs, so results do not depend on grid shape.
//
// Tile 128x128x16, 256 threads, 8x8 micro-tile per thread, operands staged K-transposed in
// shared memory (conflict-free float4 reads along M/N).
#include "common.cuh"

namespace {

constexpr int BM = 128, BN = 128, BK = 16, NT = 256;

template <typename T> __device__ __forceinline__ void load4(const T* p, float* v);
template <> __device__ __forceinline__ void load4<float>(const float* p, float* v) {
  float4 a = *reinterpret_cast<const float4*>(p); v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
}
template <> __device__ __forceinline__ void load4<bf16>(const bf16* p, float* v) {
  uint2 r = *reinterpret_cast<const uint2*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
  float2 a = __bfloat1622float2(h[0]), b = __bfloat1622float2(h[1]);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

struct EpiParams {
  void* D; int64_t ldd; const float* bias; const float* aux0; int period;
};

template <int EPI, typename TO>
__device__ __forceinline__ void epi_store(const EpiParams& p, int row, int col, float acc) {
  float v = acc + (p.bias ? p.bias[col] : 0.f);
  if (EPI == MDC_EPI_BIAS) {
    reinterpret_cast<TO*>(p.D)[(int64_t)row * p.ldd + col] = from_f<TO>(v);
  } else if (EPI == MDC_EPI_BIAS_GELU) {
    reinterpret_cast<TO*>(p.D)[(int64_t)row * p.ldd + col] = from_f<TO>(gelu_erf(v));
  } else if (EPI == MDC_EPI_BIAS_RELU) {
    reinterpret_cast<TO*>(p.D)[(int64_t)row * p.ldd + col] = from_f<TO>(fmaxf(v, 0.f));
  } else if (EPI == MDC_EPI_LS_RESIDUAL) {
    float* r = reinterpret_cast<float*>(p.D) + (int64_t)row * p.ldd + col;
    *r = *r + p.aux0[col] * v;
  } else {  // MDC_EPI_PATCH
    int img = row / p.period, pp = row - img * p.period;
    reinterpret_cast<float*>(p.D)[(int64_t)(row + img + 1) * p.ldd + col] = v + p.aux0[(int64_t)pp * p.ldd + col];
  }
}

template <typename TI, typename TO, int EPI>
__global__ void __launch_bounds__(NT) gemm_simt_kernel(const TI* __restrict__ A, int64_t lda, const TI* __restrict__ W,
                                                       int64_t ldw, EpiParams ep, int M, int N, int K) {
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Ws[BK][BN + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int tx = tid % 16, ty = tid / 16;          // micro-tile: rows ty*8.., cols tx*8..
  // loader mapping: 128 rows x 4 float4 per tile = 512 float4, 2 per thread
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += BK) {
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      int idx = tid + it * NT;          // 0..511
      int r = idx >> 2, kq = (idx & 3) * 4;
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (m0 + r < M && k0 + kq < K) load4<TI>(A + (int64_t)(m0 + r) * lda + k0 + kq, v);
#pragma unroll
      for (int j = 0; j < 4; ++j) As[kq + j][r] = v[j];
      float w[4] = {0.f, 0.f, 0.f, 0.f};
      if (n0 + r < N && k0 + kq < K) load4<TI>(W + (int64_t)(n0 + r) * ldw + k0 + kq, w);
#pragma unroll
      for (int j = 0; j < 4; ++j) Ws[kq + j][r] = w[j];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[8], b[8];
      *reinterpret_cast<float4*>(a) = *reinterpret_cast<const float4*>(&As[k][ty * 8]);
      *reinterpret_cast<float4*>(a + 4) = *reinterpret_cast<const float4*>(&As[k][ty * 8 + 4]);
      *reinterpret_cast<float4*>(b) = *reinterpret_cast<const float4*>(&Ws[k][tx * 8]);
      *reinterpret_cast<float4*>(b + 4) = *reinterpret_cast<const float4*>(&Ws[k][tx * 8 + 4]);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int row = m0 + ty * 8 + i;
    if (row >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int col = n0 + tx * 8 + j;
      if (col < N) epi_store<EPI, TO>(ep, row, col, acc[i][j]);
    }
  }
}

template <typename TI, typename TO>
int launch_typed(mdc_ctx* ctx, int epilogue, const void* A, int64_t lda, const void* W, int64_t ldw, EpiParams ep,
                 int M, int N, int K, cudaStream_t s) {
  dim3 grid((N + BN - 1) / BN, (M + BM - 1) / BM), block(NT);
  const TI* a = (const TI*)A; const TI* w = (const TI*)W;
  switch (epilogue) {
    case MDC_EPI_BIAS: gemm_simt_kernel<TI, TO, MDC_EPI_BIAS><<<grid, block, 0, s>>>(a, lda, w, ldw, ep, M, N, K); break;
    case MDC_EPI_BIAS_GELU: gemm_simt_kernel<TI, TO, MDC_EPI_BIAS_GELU><<<grid, block, 0, s>>>(a, lda, w, ldw, ep, M, N, K); break;
    case MDC_EPI_BIAS_RELU: gemm_simt_kernel<TI, TO, MDC_EPI_BIAS_RELU><<<grid, block, 0, s>>>(a, lda, w, ldw, ep, M, N, K); break;
    case MDC_EPI_LS_RESIDUAL: gemm_simt_kernel<TI, TO, MDC_EPI_LS_RESIDUAL><<<grid, block, 0, s>>>(a, lda, w, ldw, ep, M, N, K); break;
    case MDC_EPI_PATCH: gemm_simt_kernel<TI, TO, MDC_EPI_PATCH><<<grid, block, 0, s>>>(a, lda, w, ldw, ep, M, N, K); break;
    default: MDC_FAIL(-2, "gemm: unknown epilogue %d", epilogue);
  }
  MDC_LAUNCH_CHECK(ctx);
  return 0;
}

}  // namespace

int gemm_simt_launch(mdc_ctx* ctx, int dtype, int epilogue, const void* A, int64_t lda, const void* W, int64_t ldw,
                     void* D, int64_t ldd, const float* bias, const float* aux0, int period, int M, int N, int K,
                     cudaStream_t s) {
  MDC_CHECK_ARG(K % 4 == 0 && lda % 4 == 0 && ldw % 4 == 0);
  const uintptr_t vec_mask = dtype == MDC_F32 ? 15 : 7;      // A and W are read four elements at a time: float4 (f32) or uint2 (bf16)
  MDC_CHECK_ARG(((uintptr_t)A & vec_mask) == 0 && ((uintptr_t)W & vec_mask) == 0);
  EpiParams ep{D, ldd, bias, aux0, period};
  if (dtype == MDC_F32) return launch_typed<float, float>(ctx, epilogue, A, lda, W, ldw, ep, M, N, K, s);
  return launch_typed<bf16, bf16>(ctx, epilogue, A, lda, W, ldw, ep, M, N, K, s);
}

extern "C" int mdc_gemm(mdc_ctx* ctx, int dtype, int epilogue, const void* A, int64_t lda, const void* W, int64_t ldw,
                        void* D, int64_t ldd, const float* bias, const float* aux0, int period, int M, int N, int K,
                        void* stream) {
  MDC_CHECK_ARG(ctx && A && W && D);
  MDC_CHECK_DEVICE(ctx);
  MDC_CHECK_ARG(dtype == MDC_F32 || dtype == MDC_BF16 || dtype == MDC_F16);
  MDC_CHECK_ARG(M >= 0 && N > 0 && K > 0);
  if (epilogue == MDC_EPI_LS_RESIDUAL) MDC_CHECK_ARG(aux0 != nullptr);
  if (epilogue == MDC_EPI_PATCH) MDC_CHECK_ARG(aux0 != nullptr && period > 0);
  if (M == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (dtype == MDC_F16) {      // IEEE-half operands and outputs: tensor-core kernel only (bias / bias+ReLU epilogues)
    MDC_CHECK_ARG(gemm_tc_supported(M, N, K, lda, ldw));
    return gemm_tc_launch(ctx, epilogue, A, lda, W, ldw, D, ldd, bias, aux0, period, M, N, K, s, 1);
  }
  if (dtype == MDC_BF16 && !ctx->gemm_backend_simt && gemm_tc_supported(M, N, K, lda, ldw))
    return gemm_tc_launch(ctx, epilogue, A, lda, W, ldw, D, ldd, bias, aux0, period, M, N, K, s);
  return gemm_simt_launch(ctx, dtype, epilogue, A, lda, W, ldw, D, ldd, bias, aux0, period, M, N, K, s);
}
