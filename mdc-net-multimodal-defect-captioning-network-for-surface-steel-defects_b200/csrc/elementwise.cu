// elementwise.cu -- bandwidth-bound pieces of the encoder: im2col for the stride-16 patch conv,
// LayerNorm, the fused encoder tail (final norm + drop cls + channel pooling + encoder_pos_embed),
// grayscale preprocessing and positional-table interpolation.  All rows are handled warp-per-row
// with 128-bit accesses; grids are sized in units of warps so every SM gets work.
#include "common.cuh"
#include "kernels.cuh"

namespace {

// ---- patches: (B,C,H,W) f32 -> [B*n, C*p*p], patch flattened (ch, dy, dx) -- timm PatchEmbed.proj as a GEMM operand
template <typename TO>
__global__ void im2col_kernel(const float* __restrict__ x, TO* __restrict__ P, int B, int C, int img, int p) {
  const int G = img / p, n = G * G, Kc = C * p * p;
  const int chunks_per_row = Kc / 8;
  int64_t total = (int64_t)B * n * chunks_per_row;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int ck = (int)(i % chunks_per_row);
    int64_t row = i / chunks_per_row;
    int b = (int)(row / n), pi = (int)(row % n);
    int r = pi / G, c = pi % G;
    int col = ck * 8;
    int ch = col / (p * p), rem = col % (p * p), dy = rem / p, dx = rem % p;
    const float* src = x + (((int64_t)b * C + ch) * img + (r * p + dy)) * img + c * p + dx;
    float v[8]; load8(src, v);
    store8(P + row * Kc + col, v);
  }
}

__global__ void set_cls_rows_kernel(float* __restrict__ h, const float* __restrict__ cls, int B, int rows_per_img, int D) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B * D) { int b = i / D, c = i % D; h[(int64_t)b * rows_per_img * D + c] = cls[c]; }
}

// ---- LayerNorm: warp per row, two-pass statistics (mean, then centred variance) like torch
template <typename TO>
__global__ void layernorm_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ w,
                                 const float* __restrict__ b, float eps, TO* __restrict__ out, int64_t ldo,
                                 int rows, int cols) {
  int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const float* xr = x + (int64_t)warp * ldx;
  float s = 0.f;
  for (int c = lane * 4; c < cols; c += 128) { float4 v = *reinterpret_cast<const float4*>(xr + c); s += (v.x + v.y) + (v.z + v.w); }
  float mean = warp_sum(s) / (float)cols;
  float q = 0.f;
  for (int c = lane * 4; c < cols; c += 128) {
    float4 v = *reinterpret_cast<const float4*>(xr + c);
    float a0 = v.x - mean, a1 = v.y - mean, a2 = v.z - mean, a3 = v.w - mean;
    q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
  }
  float rstd = 1.0f / sqrtf(warp_sum(q) / (float)cols + eps);
  TO* orow = out + (int64_t)warp * ldo;
  for (int c = lane * 4; c < cols; c += 128) {
    float4 v = *reinterpret_cast<const float4*>(xr + c);
    float4 g = *reinterpret_cast<const float4*>(w + c), bb = *reinterpret_cast<const float4*>(b + c);
    orow[c + 0] = from_f<TO>((v.x - mean) * rstd * g.x + bb.x);
    orow[c + 1] = from_f<TO>((v.y - mean) * rstd * g.y + bb.y);
    orow[c + 2] = from_f<TO>((v.z - mean) * rstd * g.z + bb.z);
    orow[c + 3] = from_f<TO>((v.w - mean) * rstd * g.w + bb.w);
  }
}

// Fast path for cols = NV * 128 <= 1024: the row lives in registers (one global read), statistics in the same two-pass order
// (mean, then centred variance), 8-byte packed stores for bf16 output.
// A warp normalises TWO rows in lockstep (both rows' loads in flight first, the two shuffle butterflies interleaved): 12 608 rows are 788
// CTAs = one wave at the kernel's occupancy instead of 1 576 CTAs = 1.33 waves, and every warp has twice the bytes in flight.  Each
// row's own operation sequence -- and so every result bit -- is what the one-row form computed.
template <typename TO, int NV>
__global__ void __launch_bounds__(256) layernorm_rows_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ w,
                                                              const float* __restrict__ b, float eps, TO* __restrict__ out, int64_t ldo, int rows) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int r0 = 2 * warp;
  if (r0 >= rows) return;
  const bool two = r0 + 1 < rows;
  const float* xr[2] = {x + (int64_t)r0 * ldx, x + (int64_t)(two ? r0 + 1 : r0) * ldx};
  float4 v[2][NV];
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int i = 0; i < NV; ++i) v[h][i] = *reinterpret_cast<const float4*>(xr[h] + i * 128 + lane * 4);
  float4 gq[NV], bq[NV];               // weight / bias requested with the rows: one memory round trip per warp instead of two
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    gq[i] = __ldg(reinterpret_cast<const float4*>(w + i * 128 + lane * 4));
    bq[i] = __ldg(reinterpret_cast<const float4*>(b + i * 128 + lane * 4));
  }
  float s[2] = {0.f, 0.f};
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int i = 0; i < NV; ++i) s[h] += (v[h][i].x + v[h][i].y) + (v[h][i].z + v[h][i].w);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s[0] += __shfl_xor_sync(0xffffffffu, s[0], o); s[1] += __shfl_xor_sync(0xffffffffu, s[1], o); }
  const float mean[2] = {s[0] / (float)(NV * 128), s[1] / (float)(NV * 128)};
  float q[2] = {0.f, 0.f};
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float a0 = v[h][i].x - mean[h], a1 = v[h][i].y - mean[h], a2 = v[h][i].z - mean[h], a3 = v[h][i].w - mean[h];
      q[h] += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { q[0] += __shfl_xor_sync(0xffffffffu, q[0], o); q[1] += __shfl_xor_sync(0xffffffffu, q[1], o); }
  const float rstd[2] = {1.0f / sqrtf(q[0] / (float)(NV * 128) + eps), 1.0f / sqrtf(q[1] / (float)(NV * 128) + eps)};
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 128 + lane * 4;
    const float4 g = gq[i], bb = bq[i];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h == 1 && !two) break;
      TO* orow = out + (int64_t)(r0 + h) * ldo;
      const float o0 = (v[h][i].x - mean[h]) * rstd[h] * g.x + bb.x, o1 = (v[h][i].y - mean[h]) * rstd[h] * g.y + bb.y;
      const float o2 = (v[h][i].z - mean[h]) * rstd[h] * g.z + bb.z, o3 = (v[h][i].w - mean[h]) * rstd[h] * g.w + bb.w;
      if constexpr (sizeof(TO) == 2) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(o0, o1), hi = __floats2bfloat162_rn(o2, o3);
        uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&lo); pk.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(orow + c) = pk;
      } else {
        *reinterpret_cast<float4*>(orow + c) = make_float4(o0, o1, o2, o3);
      }
    }
  }
}

// ---- encoder tail: final LN (eps 1e-6), drop cls (model.py:23 features[:,1:]), AdaptiveAvgPool1d over
// channels (model.py:19), + encoder_pos_embed (model.py:103-105).  Warp per patch token.
// D = NV * 128 channels pooled in adjacent pairs (AdaptiveAvgPool1d(D / 2)): the row stays in registers (one read of the residual
// stream instead of three), a lane's float4 yields two pooled outputs.  Same arithmetic as the generic kernel below.
template <typename TO, int NV>
__global__ void __launch_bounds__(256) encoder_tail_pairs_kernel(const float* __restrict__ h, const float* __restrict__ w, const float* __restrict__ b,
                                                                 float eps, const float* __restrict__ enc_pos, float* __restrict__ enc_out,
                                                                 TO* __restrict__ memory, int B, int n) {
  constexpr int D = NV * 128, OD = D / 2;
  const int lane = threadIdx.x & 31;
  const int warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (warp >= B * n) return;
  const int bi = warp / n, pi = warp % n;
  const float* xr = h + ((int64_t)bi * (n + 1) + 1 + pi) * D;
  float4 v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = *reinterpret_cast<const float4*>(xr + i * 128 + lane * 4);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  const float mean = warp_sum(s) / (float)D;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float a0 = v[i].x - mean, a1 = v[i].y - mean, a2 = v[i].z - mean, a3 = v[i].w - mean;
    q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)D + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 128 + lane * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(w + c)), bb = __ldg(reinterpret_cast<const float4*>(b + c));
    const float y0 = (v[i].x - mean) * rstd * g.x + bb.x, y1 = (v[i].y - mean) * rstd * g.y + bb.y;
    const float y2 = (v[i].z - mean) * rstd * g.z + bb.z, y3 = (v[i].w - mean) * rstd * g.w + bb.w;
    const float p0 = (0.f + y0 + y1) / 2.0f, p1 = (0.f + y2 + y3) / 2.0f;
    const int o = c >> 1;
    const int64_t oi = ((int64_t)bi * n + pi) * OD + o;
    if (enc_out) *reinterpret_cast<float2*>(enc_out + oi) = make_float2(p0, p1);
    if (memory) {
      const float2 ep = __ldg(reinterpret_cast<const float2*>(enc_pos + (int64_t)pi * OD + o));
      memory[oi] = from_f<TO>(p0 + ep.x); memory[oi + 1] = from_f<TO>(p1 + ep.y);
    }
  }
}

template <typename TO>
__global__ void encoder_tail_kernel(const float* __restrict__ h, const float* __restrict__ w, const float* __restrict__ b,
                                    float eps, const float* __restrict__ enc_pos, float* __restrict__ enc_out,
                                    TO* __restrict__ memory, int B, int n, int D, int out_dim) {
  extern __shared__ float sm[];   // warps_per_block * D
  int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int warp = blockIdx.x * (blockDim.x >> 5) + wib;
  if (warp >= B * n) return;
  int bi = warp / n, pi = warp % n;
  const float* xr = h + ((int64_t)bi * (n + 1) + 1 + pi) * D;
  float* row = sm + wib * D;
  float s = 0.f;
  for (int c = lane * 4; c < D; c += 128) { float4 v = *reinterpret_cast<const float4*>(xr + c); s += (v.x + v.y) + (v.z + v.w); }
  float mean = warp_sum(s) / (float)D;
  float q = 0.f;
  for (int c = lane * 4; c < D; c += 128) {
    float4 v = *reinterpret_cast<const float4*>(xr + c);
    float a0 = v.x - mean, a1 = v.y - mean, a2 = v.z - mean, a3 = v.w - mean;
    q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
  }
  float rstd = 1.0f / sqrtf(warp_sum(q) / (float)D + eps);
  for (int c = lane; c < D; c += 32) row[c] = (xr[c] - mean) * rstd * w[c] + b[c];
  __syncwarp();
  for (int o = lane; o < out_dim; o += 32) {
    int st = (int)(((int64_t)o * D) / out_dim);
    int en = (int)((((int64_t)(o + 1)) * D + out_dim - 1) / out_dim);
    float acc = 0.f;
    for (int c = st; c < en; ++c) acc += row[c];
    float v = acc / (float)(en - st);
    int64_t oi = ((int64_t)bi * n + pi) * out_dim + o;
    if (enc_out) enc_out[oi] = v;
    if (memory) memory[oi] = from_f<TO>(v + enc_pos[(int64_t)pi * out_dim + o]);
  }
}

template <typename TO>
__global__ void add_pos_kernel(const float* __restrict__ enc_out, const float* __restrict__ pos, TO* __restrict__ mem,
                               int64_t total, int64_t per_img) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
    mem[i] = from_f<TO>(enc_out[i] + pos[i % per_img]);
}

// ---- u8 image -> model tensor exactly as the reference's transform does it (inference_p.py:148-158, dataset.py:109-113):
//   cv2.imread(...)[..., ::-1]          BGR -> RGB (a gray image has three equal channels)
//   A.Resize(size, size)                cv2.resize(uint8, INTER_LINEAR): FIXED-POINT bilinear, result rounded to uint8
//   A.Normalize()                       float32: (v - mean*255) * (1 / (std*255)), two roundings
// The resize is integer work and is reproduced bit for bit (OpenCV imgproc/resize.cpp, 8-bit linear path): per destination
// coordinate f = (float)((d + 0.5) * scale - 0.5) with scale = 1 / (dst / src) in double, s = floor(f), coefficients
// saturate_cast<short>((1 - f) * 2048), ((f) * 2048) rounded half-to-even; in x a source index outside the row gets coefficient
// (2048, 0) on the clamped pixel, in y the two ROWS are clamped and keep their coefficients; horizontal pass in int32, vertical pass
// ((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2.  Pinned against cv2 4.13 outputs (tests/golden/case_preprocess.pt).
struct ResizeCoef { int s; int a0, a1; };

__device__ __forceinline__ ResizeCoef resize_coef(int d, int src, int dst, bool zero_outside) {
  const double scale = __ddiv_rn(1.0, __ddiv_rn((double)dst, (double)src));
  float f = __double2float_rn(__dadd_rn(__dmul_rn((double)d + 0.5, scale), -0.5));     // no fused multiply-add: OpenCV's baseline build has none
  int s = (int)floorf(f);
  f = __fsub_rn(f, (float)s);
  if (zero_outside) {
    if (s < 0) { f = 0.f; s = 0; }
    if (s >= src - 1) { f = 0.f; s = src - 1; }
  }
  ResizeCoef c;
  c.s = s;
  c.a0 = max(-32768, min(32767, __float2int_rn(__fmul_rn(__fsub_rn(1.0f, f), 2048.0f))));
  c.a1 = max(-32768, min(32767, __float2int_rn(__fmul_rn(f, 2048.0f))));
  return c;
}

// one block per (output row, image), one thread per output column; CH = 1 (gray, (B,h,w)) or 3 (BGR interleaved, (B,h,w,3))
template <int CH>
__global__ void preprocess_u8_kernel(const uint8_t* __restrict__ src, int h, int w, float* __restrict__ out, int size,
                                     float m0, float m1, float m2, float d0, float d1, float d2) {
  const int y = blockIdx.x, b = blockIdx.y;
  const ResizeCoef cy = resize_coef(y, h, size, false);
  const int y0 = min(max(cy.s, 0), h - 1), y1 = min(max(cy.s + 1, 0), h - 1);
  const uint8_t* im = src + (int64_t)b * h * w * CH;
  const float mean[3] = {m0, m1, m2}, den[3] = {d0, d1, d2};
  for (int x = threadIdx.x; x < size; x += blockDim.x) {
    const ResizeCoef cx = resize_coef(x, w, size, true);
    const int x0 = cx.s, x1 = min(cx.s + 1, w - 1);
    int v[CH];
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      const int S0 = (int)im[((int64_t)y0 * w + x0) * CH + c] * cx.a0 + (int)im[((int64_t)y0 * w + x1) * CH + c] * cx.a1;
      const int S1 = (int)im[((int64_t)y1 * w + x0) * CH + c] * cx.a0 + (int)im[((int64_t)y1 * w + x1) * CH + c] * cx.a1;
      const int r = (((cy.a0 * (S0 >> 4)) >> 16) + ((cy.a1 * (S1 >> 4)) >> 16) + 2) >> 2;
      v[c] = min(255, max(0, r));
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {           // output channel c = R,G,B; BGR input: source channel 2 - c
      const int vv = CH == 1 ? v[0] : v[CH == 1 ? 0 : 2 - c];
      out[(((int64_t)b * 3 + c) * size + y) * size + x] = __fmul_rn(__fsub_rn((float)vv, mean[c]), den[c]);
    }
  }
}

__global__ void interp_rows_kernel(const float* __restrict__ in, int n_in, float* __restrict__ out, int n_out, int dim) {
  const float scale = (float)n_in / (float)n_out;
  int total = n_out * dim;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    int r = i / dim, c = i % dim;
    float src = fmaxf(scale * ((float)r + 0.5f) - 0.5f, 0.f);
    int i0 = min((int)src, n_in - 1), i1 = i0 + (i0 < n_in - 1 ? 1 : 0);
    float l1 = src - (float)i0, l0 = 1.f - l1;
    out[i] = l0 * in[(int64_t)i0 * dim + c] + l1 * in[(int64_t)i1 * dim + c];
  }
}

inline int blocks_for(int64_t threads, int block, int sm_count) {
  int64_t b = (threads + block - 1) / block;
  int64_t cap = (int64_t)sm_count * 16;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

int k_im2col(mdc_ctx* ctx, int dtype, const float* x, void* P, int B, int C, int img, int p, cudaStream_t s) {
  MDC_CHECK_ARG(p % 8 == 0 && img % p == 0 && img % 4 == 0);
  int64_t total = (int64_t)B * (img / p) * (img / p) * (C * p * p / 8);
  int grid = blocks_for(total, 256, ctx->sm_count);
  if (dtype == MDC_F32) im2col_kernel<float><<<grid, 256, 0, s>>>(x, (float*)P, B, C, img, p);
  else im2col_kernel<bf16><<<grid, 256, 0, s>>>(x, (bf16*)P, B, C, img, p);
  MDC_LAUNCH_CHECK(ctx); return 0;
}

int k_set_cls_rows(mdc_ctx* ctx, float* h, const float* cls, int B, int rows_per_img, int D, cudaStream_t s) {
  set_cls_rows_kernel<<<(B * D + 255) / 256, 256, 0, s>>>(h, cls, B, rows_per_img, D);
  MDC_LAUNCH_CHECK(ctx); return 0;
}

int k_encoder_tail(mdc_ctx* ctx, int dtype, const float* h, const float* w, const float* b, float eps, const float* enc_pos,
                   float* enc_out, void* memory, int B, int n, int D, int out_dim, cudaStream_t s) {
  MDC_CHECK_ARG(D % 4 == 0);
  const int wpb = 8;
  int grid = (B * n + wpb - 1) / wpb;
  size_t smem = (size_t)wpb * D * sizeof(float);
  if (D == 512 && out_dim == 256) {       // deit3_medium -> 256: rows in registers, one pass over the residual stream
    if (dtype == MDC_F32) encoder_tail_pairs_kernel<float, 4><<<grid, wpb * 32, 0, s>>>(h, w, b, eps, enc_pos, enc_out, (float*)memory, B, n);
    else encoder_tail_pairs_kernel<bf16, 4><<<grid, wpb * 32, 0, s>>>(h, w, b, eps, enc_pos, enc_out, (bf16*)memory, B, n);
    MDC_LAUNCH_CHECK(ctx); return 0;
  }
  if (dtype == MDC_F32) encoder_tail_kernel<float><<<grid, wpb * 32, smem, s>>>(h, w, b, eps, enc_pos, enc_out, (float*)memory, B, n, D, out_dim);
  else encoder_tail_kernel<bf16><<<grid, wpb * 32, smem, s>>>(h, w, b, eps, enc_pos, enc_out, (bf16*)memory, B, n, D, out_dim);
  MDC_LAUNCH_CHECK(ctx); return 0;
}

int k_add_pos(mdc_ctx* ctx, int dtype, const float* enc_out, const float* pos, void* mem, int64_t total, int64_t per_img, cudaStream_t s) {
  int grid = blocks_for(total, 256, ctx->sm_count);
  if (dtype == MDC_F32) add_pos_kernel<float><<<grid, 256, 0, s>>>(enc_out, pos, (float*)mem, total, per_img);
  else add_pos_kernel<bf16><<<grid, 256, 0, s>>>(enc_out, pos, (bf16*)mem, total, per_img);
  MDC_LAUNCH_CHECK(ctx); return 0;
}

extern "C" int mdc_layernorm(mdc_ctx* ctx, const float* x, int64_t ldx, const float* w, const float* b, float eps,
                             void* out, int64_t ldo, int out_dtype, int rows, int cols, void* stream) {
  MDC_CHECK_ARG(ctx && x && w && b && out);
  MDC_CHECK_DEVICE(ctx);
  MDC_CHECK_ARG(cols % 4 == 0 && ldx % 4 == 0 && rows >= 0);
  // both kernels read x, w and b as float4
  MDC_CHECK_ARG(((uintptr_t)x & 15) == 0 && ((uintptr_t)w & 15) == 0 && ((uintptr_t)b & 15) == 0);
  if (rows == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  int grid = (rows + 7) / 8;
  const bool vec_ok = ldo % 4 == 0 && ((uintptr_t)out & 15) == 0;     // vector stores (fast path) or scalar stores (generic kernel)
#define MDC_LN_FAST(NV_)                                                                                                        \
  if (vec_ok && cols == NV_ * 128) {                                                                                            \
    const int grid2 = (rows + 15) / 16;           /* two rows per warp */                                                        \
    if (out_dtype == MDC_F32) layernorm_rows_kernel<float, NV_><<<grid2, 256, 0, s>>>(x, ldx, w, b, eps, (float*)out, ldo, rows);  \
    else if (out_dtype == MDC_BF16) layernorm_rows_kernel<bf16, NV_><<<grid2, 256, 0, s>>>(x, ldx, w, b, eps, (bf16*)out, ldo, rows); \
    else MDC_FAIL(-2, "layernorm: bad out_dtype %d", out_dtype);                                                                \
    MDC_LAUNCH_CHECK(ctx); return 0;                                                                                            \
  }
  MDC_LN_FAST(3) MDC_LN_FAST(4) MDC_LN_FAST(6) MDC_LN_FAST(8)      // deit3 small / medium / base / large widths
#undef MDC_LN_FAST
  if (out_dtype == MDC_F32) layernorm_kernel<float><<<grid, 256, 0, s>>>(x, ldx, w, b, eps, (float*)out, ldo, rows, cols);
  else if (out_dtype == MDC_BF16) layernorm_kernel<bf16><<<grid, 256, 0, s>>>(x, ldx, w, b, eps, (bf16*)out, ldo, rows, cols);
  else MDC_FAIL(-2, "layernorm: bad out_dtype %d", out_dtype);
  MDC_LAUNCH_CHECK(ctx); return 0;
}

// A.Normalize() constants as albumentations computes them (functional.normalize): float32 mean * 255, reciprocal of float32 std * 255
static void normalize_constants(float (&m)[3], float (&d)[3]) {
  const float mean[3] = {0.485f, 0.456f, 0.406f}, sd[3] = {0.229f, 0.224f, 0.225f};
  for (int c = 0; c < 3; ++c) { m[c] = mean[c] * 255.0f; const float s = sd[c] * 255.0f; d[c] = 1.0f / s; }
}

static int preprocess_launch(mdc_ctx* ctx, const uint8_t* src, int B, int h, int w, int ch, float* out, int size, void* stream) {
  MDC_CHECK_ARG(ctx && src && out && B >= 0 && h > 0 && w > 0 && size > 0 && h < 32768 && w < 32768 && B < 65536);
  MDC_CHECK_DEVICE(ctx);
  if (B == 0) return 0;
  float m[3], d[3]; normalize_constants(m, d);
  const dim3 grid(size, B); const int block = size < 256 ? ((size + 31) / 32) * 32 : 256;
  if (ch == 1) preprocess_u8_kernel<1><<<grid, block, 0, (cudaStream_t)stream>>>(src, h, w, out, size, m[0], m[1], m[2], d[0], d[1], d[2]);
  else preprocess_u8_kernel<3><<<grid, block, 0, (cudaStream_t)stream>>>(src, h, w, out, size, m[0], m[1], m[2], d[0], d[1], d[2]);
  MDC_LAUNCH_CHECK(ctx); return 0;
}

extern "C" int mdc_preprocess_gray(mdc_ctx* ctx, const uint8_t* gray, int B, int h, int w, float* out, int size, void* stream) {
  return preprocess_launch(ctx, gray, B, h, w, 1, out, size, stream);
}

extern "C" int mdc_preprocess_bgr(mdc_ctx* ctx, const uint8_t* bgr, int B, int h, int w, float* out, int size, void* stream) {
  return preprocess_launch(ctx, bgr, B, h, w, 3, out, size, stream);
}

extern "C" int mdc_interp_rows(mdc_ctx* ctx, const float* in, int n_in, float* out, int n_out, int dim, void* stream) {
  MDC_CHECK_ARG(ctx && in && out && n_in > 0 && n_out > 0 && dim > 0);
  MDC_CHECK_DEVICE(ctx);
  int grid = blocks_for((int64_t)n_out * dim, 256, ctx->sm_count);
  interp_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(in, n_in, out, n_out, dim);
  MDC_LAUNCH_CHECK(ctx); return 0;
}
