// prefill.cu -- teacher-forced decoder pass over ALL positions at once (SURVEY 8f row 3): Decoder.forward (model.py:58-88) and
// Decoder.predict (model.py:92-127) feed a whole target sequence through nn.TransformerDecoder; nothing in them is sequential
// except the causal mask.  The autoregressive kernel (decode_cluster.cu) would run them as n dependent steps; here every layer is
//   qkv   = x . W_in^T + b                      tcgen05 GEMM over the B*n rows (fp16 operands: the decode-loop weights, DESIGN 3.7)
//   self  = softmax(q k^T / sqrt(hd) + causal + 1.0 * [key is PAD]) v      prefill_attn_kernel (mma.sync flash-style, hd = 32 / 64 / 128)
//   x     = LN1(x + self . W_o^T + b)           tcgen05 GEMM + add_layernorm_kernel
//   cross = softmax(q' K_mem^T / sqrt(hd)) V_mem over the resident cross-K/V (bf16)    prefill_attn_kernel
//   x     = LN2(x + cross . W_co^T + b);  x = LN3(x + W2 relu(W1 x + b1) + b2)
// and the vocabulary head runs once over all rows.  Mask semantics as the reference builds them (utils.py:7-12,26-30; Q7): -inf above
// the diagonal, +1.0 (a float mask, not -inf) on PAD keys.
#include "common.cuh"
#include <cuda_fp16.h>

namespace {

// ---- embedding + positional table; PAD-key bias -------------------------------------------------------------------------
__global__ void prefill_embed_kernel(const int32_t* __restrict__ tokens, int tokens_ld, int n, int dim, const float* __restrict__ emb,
                                     const float* __restrict__ pos, int pad_idx, float* __restrict__ x32, __half* __restrict__ x16,
                                     float* __restrict__ kbias, int64_t rows) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31, b = (int)(row / n), i = (int)(row % n);
  const int tok = tokens[(int64_t)b * tokens_ld + i];
  if (lane == 0) kbias[row] = tok == pad_idx ? 1.0f : 0.0f;
  for (int c = lane; c < dim; c += 32) {
    const float v = emb[(int64_t)tok * dim + c] + pos[(int64_t)i * dim + c];
    x32[row * dim + c] = v;
    x16[row * dim + c] = f16_sat(v);
  }
}

// ---- x = LayerNorm(x + y): fp32 residual stream in place + fp16 copy for the next GEMM; one warp per row, dim = 256 NV ------------
template <int NV>
__global__ void add_layernorm_kernel(float* __restrict__ x32, const __half* __restrict__ y16, const float* __restrict__ w, const float* __restrict__ bia,
                                     __half* __restrict__ x16, int64_t rows, float eps) {
  constexpr int DIM = 256 * NV;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  float v[NV][8]; float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int64_t at = row * DIM + i * 256 + lane * 8;
    const float4 a0 = *reinterpret_cast<const float4*>(x32 + at), a1 = *reinterpret_cast<const float4*>(x32 + at + 4);
    float yv[8]; load8(y16 + at, yv);
    v[i][0] = a0.x + yv[0]; v[i][1] = a0.y + yv[1]; v[i][2] = a0.z + yv[2]; v[i][3] = a0.w + yv[3];
    v[i][4] = a1.x + yv[4]; v[i][5] = a1.y + yv[5]; v[i][6] = a1.z + yv[6]; v[i][7] = a1.w + yv[7];
#pragma unroll
    for (int j = 0; j < 8; ++j) s += v[i][j];
  }
  const float mean = warp_sum(s) * (1.0f / (float)DIM);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) { const float d = v[i][j] - mean; q += d * d; }
  const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / (float)DIM) + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c0 = i * 256 + lane * 8;
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = (v[i][j] - mean) * rstd * __ldg(w + c0 + j) + __ldg(bia + c0 + j);
    store8(x32 + row * DIM + c0, o);
    uint4 h; uint32_t* hp = reinterpret_cast<uint32_t*>(&h);
#pragma unroll
    for (int j = 0; j < 4; ++j) hp[j] = pack_f16x2_sat(o[2 * j], o[2 * j + 1]);
    *reinterpret_cast<uint4*>(x16 + row * DIM + c0) = h;
  }
}

// ---- attention, head width 32 / 64 / 128, on the tensor cores ----------------------------------------------------------------------------
template <typename T> struct Mma;
template <> struct Mma<__half> {
  static __device__ __forceinline__ void mma(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) { mma_m16n8k16<__half>(c, a, b0, b1); }
  static __device__ __forceinline__ uint32_t pack(float a, float b) { return pack_f16x2(a, b); }
  static __device__ __forceinline__ uint32_t from_half2(uint32_t v) { return v; }
};
template <> struct Mma<bf16> {
  static __device__ __forceinline__ void mma(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) { mma_m16n8k16<bf16>(c, a, b0, b1); }
  static __device__ __forceinline__ uint32_t pack(float a, float b) { return pack_bf16x2(a, b); }
  static __device__ __forceinline__ uint32_t from_half2(uint32_t v) {      // the fp16 query meets bf16 keys: rounded to the cache precision
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&v));
    return pack(f.x, f.y);
  }
};

constexpr int QCH = 128;                 // queries per CTA (8 warps x 16)
template <int HD> struct AttnCfg { static constexpr int KCH = HD == 128 ? 64 : 128; };    // keys staged per chunk: K and V panels of 8-16 KB each

// One CTA = (head, image, chunk of <= 128 queries).  q: fp16 rows (b*Lq + i), k / v: TKV rows (b*Lk + j); the head's HD channels
// start at column head*HD of every operand.  kbias: f32 [B, Lk] additive key bias in natural-log units (PAD keys: +1.0) or null.
template <typename TKV, bool CAUSAL, int HD>
__global__ void __launch_bounds__(256) prefill_attn_kernel(const __half* __restrict__ q, int64_t ldq, const TKV* __restrict__ k, const TKV* __restrict__ v,
                                                           int64_t ldkv, const float* __restrict__ kbias, __half* __restrict__ out, int64_t ldo,
                                                           int Lq, int Lk, float scale_log2e) {
  constexpr int KCH = AttnCfg<HD>::KCH, CPR = HD / 8, NKS = HD / 16, NDT = HD / 8;   // chunks per row, k-steps of q.k^T, 8-wide dim tiles of o
  __shared__ __align__(128) uint8_t Ks[KCH * HD * 2];
  __shared__ __align__(128) uint8_t Vs[KCH * HD * 2];
  const int head = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, q4 = lane & 3;
  const uint32_t ks = smem_u32(Ks), vs = smem_u32(Vs);
  const int q0 = blockIdx.z * QCH + warp * 16, r0 = q0 + g, r1 = r0 + 8;
  const bool active = q0 < Lq;
  uint32_t qa[NKS][4];
#pragma unroll
  for (int s2 = 0; s2 < NKS; ++s2) {
    const __half* p0 = q + ((int64_t)b * Lq + r0) * ldq + head * HD + s2 * 16 + 2 * q4;
    const __half* p1 = q + ((int64_t)b * Lq + r1) * ldq + head * HD + s2 * 16 + 2 * q4;
    qa[s2][0] = r0 < Lq ? Mma<TKV>::from_half2(*reinterpret_cast<const uint32_t*>(p0)) : 0u;
    qa[s2][1] = r1 < Lq ? Mma<TKV>::from_half2(*reinterpret_cast<const uint32_t*>(p1)) : 0u;
    qa[s2][2] = r0 < Lq ? Mma<TKV>::from_half2(*reinterpret_cast<const uint32_t*>(p0 + 8)) : 0u;
    qa[s2][3] = r1 < Lq ? Mma<TKV>::from_half2(*reinterpret_cast<const uint32_t*>(p1 + 8)) : 0u;
  }
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  float o[NDT][4];
#pragma unroll
  for (int i = 0; i < NDT; ++i) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }
  const int k_end = CAUSAL ? min(Lk, blockIdx.z * QCH + QCH) : Lk;      // causal: no key beyond the CTA's last query
  for (int kc0 = 0; kc0 < k_end; kc0 += KCH) {
    if (kc0 > 0) __syncthreads();
    for (int i = tid; i < KCH * CPR; i += blockDim.x) {
      const int r = i / CPR, c = i % CPR, key = kc0 + r;
      if (key < Lk) {
        cp_async16(ks + swz<HD>(r, c), k + ((int64_t)b * Lk + key) * ldkv + head * HD + c * 8);
        cp_async16(vs + swz<HD>(r, c), v + ((int64_t)b * Lk + key) * ldkv + head * HD + c * 8);
      } else {
        *reinterpret_cast<uint4*>(Ks + swz<HD>(r, c)) = make_uint4(0, 0, 0, 0);
        *reinterpret_cast<uint4*>(Vs + swz<HD>(r, c)) = make_uint4(0, 0, 0, 0);
      }
    }
    cp_async_wait_all();
    __syncthreads();
    int nblk = active ? (min(KCH, Lk - kc0) + 15) / 16 : 0;
    if (CAUSAL && active) nblk = max(0, min(nblk, (q0 + 15 - kc0) / 16 + 1));     // key blocks that hold a key <= the warp's last query
    for (int kb = 0; kb < nblk; ++kb) {
      const int lk0 = kb * 16, key0 = kc0 + lk0;
      float s[2][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}};
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        const int r = lk0 + nt * 8 + (lane & 7);
#pragma unroll
        for (int kg = 0; kg < NKS / 2; ++kg) {       // 32 channels (two k-steps) per ldmatrix.x4
          uint32_t kf[4];
          ldsm_x4(kf, ks + swz<HD>(r, 4 * kg + (lane >> 3)));
          Mma<TKV>::mma(s[nt], qa[2 * kg], kf[0], kf[1]);
          Mma<TKV>::mma(s[nt], qa[2 * kg + 1], kf[2], kf[3]);
        }
      }
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = key0 + nt * 8 + 2 * q4 + (e & 1), row = (e < 2) ? r0 : r1;
          float x = s[nt][e] * scale_log2e;
          if (kbias != nullptr && key < Lk) x = fmaf(kbias[(int64_t)b * Lk + key], LOG2E, x);
          if (key >= Lk || (CAUSAL && key > row)) x = -INFINITY;
          s[nt][e] = x;
        }
      float mx0 = fmaxf(fmaxf(s[0][0], s[0][1]), fmaxf(s[1][0], s[1][1]));
      float mx1 = fmaxf(fmaxf(s[0][2], s[0][3]), fmaxf(s[1][2], s[1][3]));
      mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
      mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
      // a row can be fully masked in a block (causal, row < key0; padded query rows): keep the state untouched then
      const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
      const float c0 = mn0 == -INFINITY ? 1.f : ex2_approx(m0 - mn0), c1 = mn1 == -INFINITY ? 1.f : ex2_approx(m1 - mn1);
      const float ms0 = mn0 == -INFINITY ? 0.f : mn0, ms1 = mn1 == -INFINITY ? 0.f : mn1;
      m0 = mn0; m1 = mn1;
      float p[2][4];
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        p[nt][0] = ex2_approx(s[nt][0] - ms0); p[nt][1] = ex2_approx(s[nt][1] - ms0);
        p[nt][2] = ex2_approx(s[nt][2] - ms1); p[nt][3] = ex2_approx(s[nt][3] - ms1);
      }
      l0 = l0 * c0 + (p[0][0] + p[0][1]) + (p[1][0] + p[1][1]);
      l1 = l1 * c1 + (p[0][2] + p[0][3]) + (p[1][2] + p[1][3]);
#pragma unroll
      for (int i = 0; i < NDT; ++i) { o[i][0] *= c0; o[i][1] *= c0; o[i][2] *= c1; o[i][3] *= c1; }
      uint32_t pa[4];
      pa[0] = Mma<TKV>::pack(p[0][0], p[0][1]); pa[1] = Mma<TKV>::pack(p[0][2], p[0][3]);
      pa[2] = Mma<TKV>::pack(p[1][0], p[1][1]); pa[3] = Mma<TKV>::pack(p[1][2], p[1][3]);
#pragma unroll
      for (int dp = 0; dp < NDT / 2; ++dp) {     // two 8-wide dim tiles per ldmatrix.x4.trans
        uint32_t vf[4];
        const int r = lk0 + (lane & 7) + ((lane >> 3) & 1) * 8;
        ldsm_x4_trans(vf, vs + swz<HD>(r, dp * 2 + (lane >> 4)));
        Mma<TKV>::mma(o[2 * dp], pa, vf[0], vf[1]);
        Mma<TKV>::mma(o[2 * dp + 1], pa, vf[2], vf[3]);
      }
    }
  }
  if (!active) return;
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.0f / l0, i1 = 1.0f / l1;
  __half* ob = out + ((int64_t)b * Lq) * ldo + head * HD + 2 * q4;
#pragma unroll
  for (int nt = 0; nt < NDT; ++nt) {
    if (r0 < Lq) *reinterpret_cast<__half2*>(ob + (int64_t)r0 * ldo + nt * 8) = __floats2half2_rn(o[nt][0] * i0, o[nt][1] * i0);
    if (r1 < Lq) *reinterpret_cast<__half2*>(ob + (int64_t)r1 * ldo + nt * 8) = __floats2half2_rn(o[nt][2] * i1, o[nt][3] * i1);
  }
}

// ---- vocabulary head over all rows: logits f32 = x16 . W^T + b (fp16 operands, fp32 accumulation, as the decode kernel's head) ----
constexpr int HEAD_ROWS = 8;
__global__ void __launch_bounds__(128) prefill_head_kernel(const __half* __restrict__ x16, const __half* __restrict__ W, const float* __restrict__ bias,
                                                           float* __restrict__ logits, int64_t img_stride, int row_offset, int n, int n_out, int V,
                                                           int64_t rows, int dim) {
  extern __shared__ __align__(16) float head_xs[];          // [HEAD_ROWS][dim]
  const int64_t row0 = (int64_t)blockIdx.x * HEAD_ROWS;
  for (int i = threadIdx.x; i < HEAD_ROWS * dim; i += blockDim.x) {
    const int r = i / dim, c = i - r * dim;
    head_xs[i] = row0 + r < rows ? __half2float(x16[(row0 + r) * dim + c]) : 0.f;
  }
  __syncthreads();
  for (int vb = threadIdx.x; vb < V; vb += blockDim.x) {
    float acc[HEAD_ROWS];
#pragma unroll
    for (int r = 0; r < HEAD_ROWS; ++r) acc[r] = 0.f;
    const __half* wr = W + (int64_t)vb * dim;
    for (int c = 0; c < dim; c += 8) {
      float wv[8]; load8(wr + c, wv);
#pragma unroll
      for (int r = 0; r < HEAD_ROWS; ++r)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[r] = fmaf(wv[j], head_xs[r * dim + c + j], acc[r]);
    }
    const float bv = bias[vb];
#pragma unroll
    for (int r = 0; r < HEAD_ROWS; ++r) {
      const int64_t row = row0 + r;
      if (row < rows) {
        const int b = (int)(row / n), i = (int)(row % n);
        if (i < n_out) logits[(int64_t)b * img_stride + (int64_t)(i + row_offset) * V + vb] = acc[r] + bv;
      }
    }
  }
}

struct Ws { float* x32; __half* x16; __half* qkv; __half* o16; __half* y16; __half* h16; float* kbias; };

size_t ws_bytes(const mdc_dims& d, int B, int n) {
  const size_t R = (size_t)B * n;
  return align_up(R * d.dim * 4, 256) + align_up(R * d.dim * 2, 256) + align_up(R * 3 * d.dim * 2, 256) + align_up(R * d.dim * 2, 256) +
         align_up(R * d.dim * 2, 256) + align_up(R * d.dec_ffn * 2, 256) + align_up(R * 4, 256);
}

bool geometry_ok(const mdc_dims& d) {
  const int hd = d.dec_heads > 0 ? d.dim / d.dec_heads : 0;
  return d.precision == MDC_BF16 && (d.dim == 256 || d.dim == 512 || d.dim == 1024) && hd * d.dec_heads == d.dim &&
         (hd == 32 || hd == 64 || hd == 128) && d.dec_ffn % 8 == 0 && d.dec_layers >= 1;
}

}  // namespace

extern "C" size_t mdc_decoder_prefill_workspace_bytes(const mdc_model* m, int B, int n) {
  if (!m || B <= 0 || n <= 0 || !geometry_ok(m->d)) return 0;
  return ws_bytes(m->d, B, n);
}

extern "C" int mdc_decoder_prefill(mdc_model* m, const int32_t* tokens, int tokens_ld, int B, int n, const float* pos, const void* cross_kv,
                                   float* logits, int logits_ld, int row_offset, int n_out, void* workspace, size_t workspace_bytes, void* stream) {
  MDC_CHECK_ARG(m && tokens && cross_kv && logits && workspace && B > 0 && n > 0 && tokens_ld >= n);
  MDC_CHECK_DEVICE(m->ctx);
  MDC_CHECK_ARG(geometry_ok(m->d));
  MDC_CHECK_ARG(workspace_bytes >= ws_bytes(m->d, B, n));
  MDC_CHECK_ARG(n_out >= 0 && n_out <= n && row_offset >= 0 && n_out + row_offset <= logits_ld);
  mdc_ctx* ctx = m->ctx; const mdc_dims& d = m->d; cudaStream_t s = (cudaStream_t)stream;
  const int dim = d.dim, S = d.n_patches, heads = d.dec_heads;
  const void** gw = m->w + MDC_ENC_GLOBAL_SLOTS + d.enc_depth * MDC_ENC_BLOCK_SLOTS;
  const void** lw0 = gw + MDC_DEC_GLOBAL_SLOTS;
  if (!pos) { MDC_CHECK_ARG(n <= d.max_pos); pos = (const float*)gw[MDC_DEC_POS]; }
  const int64_t R = (int64_t)B * n;
  char* p = (char*)workspace; Ws w;
  w.x32 = (float*)p; p += align_up(R * dim * 4, 256);
  w.x16 = (__half*)p; p += align_up(R * dim * 2, 256);
  w.qkv = (__half*)p; p += align_up(R * 3 * dim * 2, 256);
  w.o16 = (__half*)p; p += align_up(R * dim * 2, 256);
  w.y16 = (__half*)p; p += align_up(R * dim * 2, 256);
  w.h16 = (__half*)p; p += align_up(R * d.dec_ffn * 2, 256);
  w.kbias = (float*)p;
  const int rows_per_block = 8;
  const int row_blocks = (int)((R + rows_per_block - 1) / rows_per_block);
  prefill_embed_kernel<<<row_blocks, rows_per_block * 32, 0, s>>>(tokens, tokens_ld, n, dim, (const float*)gw[MDC_EMB], pos, d.pad_idx, w.x32, w.x16, w.kbias, R);
  MDC_LAUNCH_CHECK(ctx);
  const int hd = dim / heads;
  const float scale_log2e = LOG2E / sqrtf((float)hd);
  const dim3 agrid(heads, B, (n + QCH - 1) / QCH);
#define MDC_ATTN(TKV_, CAUSAL_, ...)                                                                          \
  {                                                                                                           \
    if (hd == 32) prefill_attn_kernel<TKV_, CAUSAL_, 32><<<agrid, 256, 0, s>>>(__VA_ARGS__);                  \
    else if (hd == 64) prefill_attn_kernel<TKV_, CAUSAL_, 64><<<agrid, 256, 0, s>>>(__VA_ARGS__);             \
    else prefill_attn_kernel<TKV_, CAUSAL_, 128><<<agrid, 256, 0, s>>>(__VA_ARGS__);                          \
    MDC_LAUNCH_CHECK(ctx);                                                                                    \
  }
#define MDC_ADDLN(...)                                                                                        \
  {                                                                                                           \
    if (dim == 256) add_layernorm_kernel<1><<<row_blocks, rows_per_block * 32, 0, s>>>(__VA_ARGS__);          \
    else if (dim == 512) add_layernorm_kernel<2><<<row_blocks, rows_per_block * 32, 0, s>>>(__VA_ARGS__);     \
    else add_layernorm_kernel<4><<<row_blocks, rows_per_block * 32, 0, s>>>(__VA_ARGS__);                     \
    MDC_LAUNCH_CHECK(ctx);                                                                                    \
  }
  for (int l = 0; l < d.dec_layers; ++l) {
    const void** lw = lw0 + l * MDC_DEC_LAYER_SLOTS;
    // self-attention block
    MDC_TRY(mdc_gemm(ctx, MDC_F16, MDC_EPI_BIAS, w.x16, dim, lw[MDC_SA_IN_W], dim, w.qkv, 3 * dim, (const float*)lw[MDC_SA_IN_B], nullptr, 0, (int)R, 3 * dim, dim, s));
    MDC_ATTN(__half, true, w.qkv, 3 * dim, w.qkv + dim, w.qkv + 2 * dim, 3 * dim, w.kbias, w.o16, dim, n, n, scale_log2e)
    MDC_TRY(mdc_gemm(ctx, MDC_F16, MDC_EPI_BIAS, w.o16, dim, lw[MDC_SA_OUT_W], dim, w.y16, dim, (const float*)lw[MDC_SA_OUT_B], nullptr, 0, (int)R, dim, dim, s));
    MDC_ADDLN(w.x32, w.y16, (const float*)lw[MDC_LN1_W], (const float*)lw[MDC_LN1_B], w.x16, R, 1e-5f)
    // cross-attention block: q from rows [0,dim) of the packed in-projection; K/V = the resident cross-K/V of this layer
    MDC_TRY(mdc_gemm(ctx, MDC_F16, MDC_EPI_BIAS, w.x16, dim, lw[MDC_CA_IN_W], dim, w.qkv, dim, (const float*)lw[MDC_CA_IN_B], nullptr, 0, (int)R, dim, dim, s));
    const bf16* ckv = (const bf16*)cross_kv + (size_t)l * B * S * 2 * dim;
    MDC_ATTN(bf16, false, w.qkv, dim, ckv, ckv + dim, 2 * dim, nullptr, w.o16, dim, n, S, scale_log2e)
    MDC_TRY(mdc_gemm(ctx, MDC_F16, MDC_EPI_BIAS, w.o16, dim, lw[MDC_CA_OUT_W], dim, w.y16, dim, (const float*)lw[MDC_CA_OUT_B], nullptr, 0, (int)R, dim, dim, s));
    MDC_ADDLN(w.x32, w.y16, (const float*)lw[MDC_LN2_W], (const float*)lw[MDC_LN2_B], w.x16, R, 1e-5f)
    // feed-forward block
    MDC_TRY(mdc_gemm(ctx, MDC_F16, MDC_EPI_BIAS_RELU, w.x16, dim, lw[MDC_FF1_W], dim, w.h16, d.dec_ffn, (const float*)lw[MDC_FF1_B], nullptr, 0, (int)R, d.dec_ffn, dim, s));
    MDC_TRY(mdc_gemm(ctx, MDC_F16, MDC_EPI_BIAS, w.h16, d.dec_ffn, lw[MDC_FF2_W], d.dec_ffn, w.y16, dim, (const float*)lw[MDC_FF2_B], nullptr, 0, (int)R, dim, d.dec_ffn, s));
    MDC_ADDLN(w.x32, w.y16, (const float*)lw[MDC_LN3_W], (const float*)lw[MDC_LN3_B], w.x16, R, 1e-5f)
  }
  if (n_out > 0) {
    prefill_head_kernel<<<(int)((R + HEAD_ROWS - 1) / HEAD_ROWS), 128, (size_t)HEAD_ROWS * dim * sizeof(float), s>>>(
        w.x16, (const __half*)gw[MDC_OUT_W], (const float*)gw[MDC_OUT_B], logits, (int64_t)logits_ld * d.vocab, row_offset, n, n_out, d.vocab, R, dim);
    MDC_LAUNCH_CHECK(ctx);
  }
#undef MDC_ATTN
#undef MDC_ADDLN
  return 0;
}
