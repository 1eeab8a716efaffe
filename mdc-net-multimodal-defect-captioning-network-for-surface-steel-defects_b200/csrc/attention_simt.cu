// attention_simt.cu -- strip attention, fp32 arithmetic (north_star (b): "fused kernel that stages
// each row or column strip in shared memory, with warp-shuffle softmax").
//
// One CTA = (strip, head, block of 32 queries).  Keys/values of the strip stream through shared
// memory in tiles of 64 keys (K transposed so that lane == key is conflict-free); each warp owns 8
// queries and runs an online softmax whose max / sum reductions are warp shuffles.  Probabilities
// never touch memory: they are broadcast lane-to-lane with shuffles for the P.V product.
// Serves AxialAttention (axial_model.py:28-40), the ViT blocks' attention (timm Attention) and
// 14-token row/column strips; element type float (exact path) or bf16 (storage only, fp32 math).
#include "common.cuh"

namespace {

constexpr int QB = 32;      // queries per CTA
constexpr int KT = 64;      // keys per tile
constexpr int NW = 4;       // warps per CTA
constexpr int QW = QB / NW; // queries per warp (8), processed 4 at a time

template <typename T, int HD>
__global__ void __launch_bounds__(NW * 32) strip_attn_kernel(const T* __restrict__ qkv, int64_t ld, T* __restrict__ out,
                                                             int64_t ldo, int strip_len, int heads, float scale) {
  extern __shared__ __align__(16) float smem_f[];
  float (*KsT)[KT] = reinterpret_cast<float (*)[KT]>(smem_f);                 // [HD][KT]
  float (*Vs)[HD] = reinterpret_cast<float (*)[HD]>(smem_f + HD * KT);        // [KT][HD]
  float (*Qs)[HD] = reinterpret_cast<float (*)[HD]>(smem_f + 2 * HD * KT);    // [QB][HD]
  constexpr int DPL = HD / 32;   // output channels per lane
  const int strip = blockIdx.z, head = blockIdx.y, q0 = blockIdx.x * QB;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D = heads * HD;
  const T* base = qkv + (int64_t)strip * strip_len * ld + head * HD;

  // stage the query block (pre-scaled like timm: q * scale; for AxialAttention dots * scale -- the
  // product is associative up to one rounding, accounted for in the stated tolerance)
  for (int i = tid; i < QB * (HD / 8); i += NW * 32) {
    int r = i / (HD / 8), c = (i % (HD / 8)) * 8;
    float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (q0 + r < strip_len) load8(base + (int64_t)(q0 + r) * ld + c, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) Qs[r][c + j] = v[j];
  }

  float m[QW], l[QW], acc[QW][DPL];
#pragma unroll
  for (int i = 0; i < QW; ++i) { m[i] = -INFINITY; l[i] = 0.f;
#pragma unroll
    for (int j = 0; j < DPL; ++j) acc[i][j] = 0.f; }

  for (int k0 = 0; k0 < strip_len; k0 += KT) {
    __syncthreads();
    // K tile, transposed: consecutive lanes take consecutive keys -> conflict-free smem writes
    for (int i = tid; i < KT * (HD / 8); i += NW * 32) {
      int key = i % KT, c = (i / KT) * 8;
      float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (k0 + key < strip_len) load8(base + (int64_t)(k0 + key) * ld + D + c, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) KsT[c + j][key] = v[j];
    }
    for (int i = tid; i < KT * (HD / 8); i += NW * 32) {
      int key = i / (HD / 8), c = (i % (HD / 8)) * 8;
      float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (k0 + key < strip_len) load8(base + (int64_t)(k0 + key) * ld + 2 * D + c, v);
      *reinterpret_cast<float4*>(&Vs[key][c]) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(&Vs[key][c + 4]) = make_float4(v[4], v[5], v[6], v[7]);
    }
    __syncthreads();
    const bool valid0 = (k0 + lane) < strip_len, valid1 = (k0 + lane + 32) < strip_len;
#pragma unroll
    for (int g = 0; g < QW; g += 4) {
      // scores of 4 queries against this lane's 2 keys
      float s0[4] = {0, 0, 0, 0}, s1[4] = {0, 0, 0, 0};
#pragma unroll 8
      for (int d = 0; d < HD; ++d) {
        float ka = KsT[d][lane], kb = KsT[d][lane + 32];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float qv = Qs[warp * QW + g + i][d];
          s0[i] = fmaf(qv, ka, s0[i]); s1[i] = fmaf(qv, kb, s1[i]);
        }
      }
      float p0[4], p1[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a = valid0 ? s0[i] * scale : -INFINITY, b = valid1 ? s1[i] * scale : -INFINITY;
        float mn = fmaxf(m[g + i], warp_max(fmaxf(a, b)));
        float corr = expf(m[g + i] - mn);
        p0[i] = expf(a - mn); p1[i] = expf(b - mn);
        l[g + i] = l[g + i] * corr + warp_sum(p0[i] + p1[i]);
        m[g + i] = mn;
#pragma unroll
        for (int j = 0; j < DPL; ++j) acc[g + i][j] *= corr;
      }
      // P.V: lane owns channels lane + 32*j; probabilities broadcast by shuffle
      const int kmax = min(KT, strip_len - k0);
      for (int key = 0; key < kmax; ++key) {
        float vv[DPL];
#pragma unroll
        for (int j = 0; j < DPL; ++j) vv[j] = Vs[key][lane + 32 * j];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float p = __shfl_sync(0xffffffffu, key < 32 ? p0[i] : p1[i], key & 31);
#pragma unroll
          for (int j = 0; j < DPL; ++j) acc[g + i][j] = fmaf(p, vv[j], acc[g + i][j]);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < QW; ++i) {
    int q = q0 + warp * QW + i;
    if (q >= strip_len) continue;
    T* o = out + ((int64_t)strip * strip_len + q) * ldo + head * HD;
    float inv = 1.0f / l[i];
#pragma unroll
    for (int j = 0; j < DPL; ++j) o[lane + 32 * j] = from_f<T>(acc[i][j] * inv);
  }
}

// softmax over the QUERY axis (AxialAttention.forward(axis=-2), axial_model.py:36): whole strip in smem.
template <typename T>
__global__ void strip_attn_colsoftmax_kernel(const T* __restrict__ qkv, int64_t ld, T* __restrict__ out, int64_t ldo,
                                             int n, int heads, int hd, float scale) {
  extern __shared__ float sm[];
  float* S = sm;                 // [n][n+1]
  float* Q = S + n * (n + 1);    // [n][hd]
  float* K = Q + n * hd;
  float* V = K + n * hd;
  const int strip = blockIdx.y, head = blockIdx.x, D = heads * hd;
  const T* base = qkv + (int64_t)strip * n * ld + head * hd;
  for (int i = threadIdx.x; i < n * hd; i += blockDim.x) {
    int r = i / hd, c = i % hd;
    Q[i] = to_f<T>(base[(int64_t)r * ld + c]);
    K[i] = to_f<T>(base[(int64_t)r * ld + D + c]);
    V[i] = to_f<T>(base[(int64_t)r * ld + 2 * D + c]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n * n; i += blockDim.x) {
    int qi = i / n, kj = i % n;
    float s = 0.f;
    for (int d = 0; d < hd; ++d) s = fmaf(Q[qi * hd + d], K[kj * hd + d], s);
    S[qi * (n + 1) + kj] = s * scale;
  }
  __syncthreads();
  for (int kj = threadIdx.x; kj < n; kj += blockDim.x) {   // normalise each column over the queries
    float mx = -INFINITY;
    for (int qi = 0; qi < n; ++qi) mx = fmaxf(mx, S[qi * (n + 1) + kj]);
    float sum = 0.f;
    for (int qi = 0; qi < n; ++qi) { float e = expf(S[qi * (n + 1) + kj] - mx); S[qi * (n + 1) + kj] = e; sum += e; }
    float inv = 1.0f / sum;
    for (int qi = 0; qi < n; ++qi) S[qi * (n + 1) + kj] *= inv;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n * hd; i += blockDim.x) {
    int qi = i / hd, d = i % hd;
    float a = 0.f;
    for (int kj = 0; kj < n; ++kj) a = fmaf(S[qi * (n + 1) + kj], V[kj * hd + d], a);
    out[((int64_t)strip * n + qi) * ldo + head * hd + d] = from_f<T>(a);
  }
}

template <typename T>
int launch_rows(mdc_ctx* ctx, const void* qkv, int64_t ld, void* out, int64_t ldo, int n_strips, int strip_len, int heads,
                int hd, float scale, cudaStream_t s) {
  dim3 grid((strip_len + QB - 1) / QB, heads, n_strips), block(NW * 32);
  const T* in = (const T*)qkv; T* o = (T*)out;
#define MDC_ATTN_CASE(H)                                                                                         \
  {                                                                                                              \
    size_t smem = (size_t)(2 * H * KT + QB * H) * sizeof(float);                                                 \
    MDC_ENSURE_SMEM((strip_attn_kernel<T, H>), smem);                                                            \
    strip_attn_kernel<T, H><<<grid, block, smem, s>>>(in, ld, o, ldo, strip_len, heads, scale);                    \
  }
  if (hd == 32) MDC_ATTN_CASE(32)
  else if (hd == 64) MDC_ATTN_CASE(64)
  else if (hd == 128) MDC_ATTN_CASE(128)
  else MDC_FAIL(-2, "strip_attention: head_dim %d not in {32,64,128}", hd);
#undef MDC_ATTN_CASE
  MDC_LAUNCH_CHECK(ctx); return 0;
}

// shared memory of strip_attn_colsoftmax_kernel: the score matrix S [n][n+1] and Q, K, V [n][hd]
size_t cols_smem_bytes(int n, int hd) { return ((size_t)n * (n + 1) + 3 * (size_t)n * hd) * sizeof(float); }

template <typename T>
int launch_cols(mdc_ctx* ctx, const void* qkv, int64_t ld, void* out, int64_t ldo, int n_strips, int n, int heads, int hd,
                float scale, cudaStream_t s) {
  const size_t smem = cols_smem_bytes(n, hd);
  MDC_ENSURE_SMEM(strip_attn_colsoftmax_kernel<T>, smem);
  strip_attn_colsoftmax_kernel<T><<<dim3(heads, n_strips), 256, smem, s>>>((const T*)qkv, ld, (T*)out, ldo, n, heads, hd, scale);
  MDC_LAUNCH_CHECK(ctx); return 0;
}

}  // namespace

int attn_tc_supported(int strip_len, int head_dim);
int attn_tc_launch(mdc_ctx* ctx, const void* qkv, int64_t ld, void* out, int64_t ldo, int n_strips, int strip_len, int heads,
                   int head_dim, float scale, cudaStream_t s);

int attn_umma_supported(int strip_len, int head_dim, int64_t ld, int64_t ldo);
int attn_umma_launch(mdc_ctx* ctx, const void* qkv, int64_t ld, void* out, int64_t ldo, int n_strips, int strip_len, int heads, float scale,
                     cudaStream_t s);

extern "C" int mdc_strip_attention(mdc_ctx* ctx, int dtype, const void* qkv, int64_t ld_qkv, void* out, int64_t ld_out,
                                   int n_strips, int strip_len, int heads, int head_dim, float scale,
                                   int softmax_over_queries, void* stream) {
  MDC_CHECK_ARG(ctx && qkv && out);
  MDC_CHECK_DEVICE(ctx);
  MDC_CHECK_ARG(dtype == MDC_F32 || dtype == MDC_BF16);
  MDC_CHECK_ARG(n_strips >= 0 && strip_len > 0 && heads > 0 && heads <= 65535 && n_strips <= 65535 * 32);
  MDC_CHECK_ARG(ld_qkv % 8 == 0 && head_dim % 8 == 0);
  MDC_CHECK_ARG(((uintptr_t)qkv & 15) == 0);     // rows of q, k and v are read in 16-byte vectors (load8, TMA)
  if (n_strips == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (softmax_over_queries) {
    MDC_CHECK_ARG(strip_len <= 128 && head_dim <= 128);
    // the whole strip is staged in shared memory: checked before any CUDA call that could fail on it
    int smem_max = 0;
    MDC_CUDA(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
    const size_t smem = cols_smem_bytes(strip_len, head_dim);
    if (smem > (size_t)smem_max)
      MDC_FAIL(-2, "strip_attention: softmax over queries stages (n(n+1) + 3 n head_dim) floats = %zu bytes of shared memory for "
                   "n = %d, head_dim = %d; a block may use at most %d bytes", smem, strip_len, head_dim, smem_max);
    return dtype == MDC_F32 ? launch_cols<float>(ctx, qkv, ld_qkv, out, ld_out, n_strips, strip_len, heads, head_dim, scale, s)
                            : launch_cols<bf16>(ctx, qkv, ld_qkv, out, ld_out, n_strips, strip_len, heads, head_dim, scale, s);
  }
  MDC_CHECK_ARG(n_strips <= 65535);
  // bf16, head width 64: strips of up to 256 tokens (the ViT's 197) on tcgen05 / TMEM / TMA (attention_umma.cu); longer strips on the
  // chunked mma.sync kernel (attention_tc.cu); everything else (fp32, other head widths) on the SIMT kernel
  if (dtype == MDC_BF16 && !ctx->attn_backend_simt && attn_umma_supported(strip_len, head_dim, ld_qkv, ld_out) && ((uintptr_t)out & 15) == 0)
    return attn_umma_launch(ctx, qkv, ld_qkv, out, ld_out, n_strips, strip_len, heads, scale, s);
  if (dtype == MDC_BF16 && !ctx->attn_backend_simt && attn_tc_supported(strip_len, head_dim))
    return attn_tc_launch(ctx, qkv, ld_qkv, out, ld_out, n_strips, strip_len, heads, head_dim, scale, s);
  return dtype == MDC_F32 ? launch_rows<float>(ctx, qkv, ld_qkv, out, ld_out, n_strips, strip_len, heads, head_dim, scale, s)
                          : launch_rows<bf16>(ctx, qkv, ld_qkv, out, ld_out, n_strips, strip_len, heads, head_dim, scale, s);
}
