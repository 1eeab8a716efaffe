// decode.cu -- one autoregressive decode step of the transformer decoder (Decoder.predict /
// nn.TransformerDecoder post-norm layers, model.py:92-127 + torch transformer.py:1158-1197),
// computed ONLY for the new position t (the reference recomputes all 99 positions and the whole
// encoder every step, SURVEY Q8/Q9).
//
// Data flow per layer (all activations f32, [B, *]; weights/KV `precision`):
//   qkv  = LNload(x) . Ws^T + bs          -> append k,v to the paged self-KV cache, slot t
//   o    = softmax(q.K[0..t]/sqrt(hd) + padbias) V[0..t]        (padbias: +1.0 at PAD keys, Q7)
//   y1   = o . Wso^T + bso
//   qc   = LNload(xa + y1; norm1) . Wcq^T + bcq
//   oc   = softmax(qc.Kc^T/sqrt(hd)) Vc   (cross K/V built once per image, HBM/L2 resident)
//   y2   = oc . Wco^T + bco
//   f1   = relu(LNload(xb + y2; norm2) . W1^T + b1)
//   y3   = f1 . W2^T + b2                 ; next layer / head consumes LNload(xc + y3; norm3)
// "LNload": residual add + LayerNorm are fused into the CONSUMER's operand load (every CTA
// re-normalises the few rows it needs; CTA column 0 also publishes the normalised rows as the
// next residual), so no projection needs a full-row epilogue and all of them spread over the SMs.
// The head kernel fuses LN3 + vocab projection + greedy / top-k / top-p select + max-prob.
// Batches of 16 and more on fp16 decode-loop weights (the wide geometry of trail_01.py:158-160 -- dim 1024, 8 x 128, 8 layers -- and the
// dim-256 geometry when the per-operation path is asked for) take a second form of the same data flow: the operand rows are built ONCE
// per linear as IEEE half (prep_x_half_vec_kernel: LayerNorm-on-load / embedding, also publishes the f32 residual), the linears are
// dec_linear_stream_kernel (weight rows as the MMA M operand, 16-32 rows per CTA, K split over the warps), the attention kernels write
// the half operand of their out-projection, and cross-attention splits the memory keys over a CTA (dec_cross_attn_split_kernel).
#include "common.cuh"
#include "select.cuh"
#include <cuda_fp16.h>
#include <float.h>
#include <type_traits>

int decode_cluster_supported(const mdc_model* m, const mdc_decode_state* st, int t_end);
int decode_cluster_launch(mdc_model* m, const mdc_decode_state* st, int t_begin, int t_end, void* logits_scratch, cudaStream_t s);

namespace {

constexpr int LIN_THREADS = 256;
constexpr int LIN_WARPS = 8;
constexpr int BT = 16;           // batch rows per CTA

enum { XMODE_PLAIN = 0, XMODE_LN = 1, XMODE_EMBED = 2, XMODE_HALF = 3 };

struct XSrc {
  int mode;
  const float* x; int64_t ldx;                  // PLAIN
  const float* resid; const float* delta;       // LN: LN(resid + delta) rows of width K
  const float* ln_w; const float* ln_b; float eps;
  const int32_t* tokens; int tokens_ld; int t;  // EMBED: emb[tokens[b,t]] + pos[t]
  const float* emb; const float* pos;
  float* xn_out;                                // where CTA column 0 publishes the operand rows (or NULL)
  const __half* xh;                             // HALF: operand rows already built as IEEE half [B][K] (prep_x_half_kernel);
                                                // PLAIN: optional IEEE-half twin of the f32 rows, written by the producer (row pitch ldxh)
  int64_t ldxh;
  const int* done;                              // stop at EOS: the batch's all-finished flag (NULL without stopping); set = return at entry
};

// stop at EOS (per-operation path): every kernel of a step returns at entry once the whole batch has finished
__device__ __forceinline__ bool batch_done(const int* done) { return done != nullptr && *done != 0; }

// ---- operand rows: LayerNorm-on-load LN(resid + delta) or embedding emb[tokens[b, t]] + pos[t], K <= MDC_MAX_DEC_DIM columns ----
// One builder per form, shared by the kernel that builds a linear's operand tile in shared memory and the one that builds the rows
// as IEEE half in global memory, so a row has the same bits whichever kernel built it.

// Scalar form, any K: lane handles the columns c = lane + 32 i < K of row b.
//   REGS : v is a register array, v[i] = column c; the loops run a constant 32 times, unroll fully, and every load is in flight at once
//   else : v is the row itself (shared memory), v[c] = column c; the loops stop at K
template <bool REGS>
__device__ __forceinline__ void operand_row(const XSrc& xs, int b, int K, float* v) {
  const int lane = threadIdx.x & 31, cend = REGS ? lane + MDC_MAX_DEC_DIM : K;
  auto at = [&](int i, int c) -> float& { return v[REGS ? i : c]; };
  if (xs.mode == XMODE_EMBED) {
    const int tok = xs.tokens[(int64_t)b * xs.tokens_ld + xs.t];
    const float* e = xs.emb + (int64_t)tok * K; const float* pz = xs.pos + (int64_t)xs.t * K;
    for (int c = lane, i = 0; c < cend; c += 32, ++i) { if (c < K) at(i, c) = e[c] + pz[c]; }
  } else {
    const float* a = xs.resid + (int64_t)b * K; const float* d = xs.delta + (int64_t)b * K;
    float sum = 0.f;
    for (int c = lane, i = 0; c < cend; c += 32, ++i) { if (c < K) { const float x = a[c] + d[c]; at(i, c) = x; sum += x; } }
    const float mean = warp_sum(sum) / (float)K;
    float q = 0.f;
    for (int c = lane, i = 0; c < cend; c += 32, ++i) { if (c < K) { const float t = at(i, c) - mean; q += t * t; } }
    const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)K + xs.eps);
    for (int c = lane, i = 0; c < cend; c += 32, ++i) { if (c < K) at(i, c) = (at(i, c) - mean) * rstd * xs.ln_w[c] + xs.ln_b[c]; }
  }
}

// Vector form, K = NV * 128: lane holds the float4 at columns 128 i + 4 lane of the R rows b + 8 h, built in lockstep; rows past the
// batch (>= B) are built from a valid row and must not be stored.  Every load of all R rows, the LayerNorm weights included, is issued
// before the first reduction: one memory round trip instead of two.
template <int NV, int R>
__device__ __forceinline__ void operand_rows_vec(const XSrc& xs, int b, int B, float4 (&v)[R][NV]) {
  static_assert(NV * 128 <= MDC_MAX_DEC_DIM, "operand rows are model rows");
  constexpr int K = NV * 128;
  const int lane = threadIdx.x & 31;
  if (xs.mode == XMODE_EMBED) {
    int tok[R];
#pragma unroll
    for (int h = 0; h < R; ++h) { const int bh = b + 8 * h; tok[h] = (bh < B) ? xs.tokens[(int64_t)bh * xs.tokens_ld + xs.t] : 0; }
    float4 pz[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) pz[i] = __ldg(reinterpret_cast<const float4*>(xs.pos + (int64_t)xs.t * K + (i * 32 + lane) * 4));
#pragma unroll
    for (int h = 0; h < R; ++h)
#pragma unroll
      for (int i = 0; i < NV; ++i) v[h][i] = __ldg(reinterpret_cast<const float4*>(xs.emb + (int64_t)tok[h] * K + (i * 32 + lane) * 4));
#pragma unroll
    for (int h = 0; h < R; ++h)
#pragma unroll
      for (int i = 0; i < NV; ++i) { v[h][i].x += pz[i].x; v[h][i].y += pz[i].y; v[h][i].z += pz[i].z; v[h][i].w += pz[i].w; }
  } else {  // XMODE_LN
    float4 dl[R][NV];
#pragma unroll
    for (int h = 0; h < R; ++h) {
      const int bh = min(b + 8 * h, B - 1);
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        v[h][i] = *reinterpret_cast<const float4*>(xs.resid + (int64_t)bh * K + (i * 32 + lane) * 4);
        dl[h][i] = *reinterpret_cast<const float4*>(xs.delta + (int64_t)bh * K + (i * 32 + lane) * 4);
      }
    }
    float4 g[NV], be[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      g[i] = __ldg(reinterpret_cast<const float4*>(xs.ln_w + (i * 32 + lane) * 4));
      be[i] = __ldg(reinterpret_cast<const float4*>(xs.ln_b + (i * 32 + lane) * 4));
    }
#pragma unroll
    for (int h = 0; h < R; ++h) {
      float sum = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        v[h][i].x += dl[h][i].x; v[h][i].y += dl[h][i].y; v[h][i].z += dl[h][i].z; v[h][i].w += dl[h][i].w;
        sum += (v[h][i].x + v[h][i].y) + (v[h][i].z + v[h][i].w);
      }
      const float mean = warp_sum(sum) / (float)K;
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        float a0 = v[h][i].x - mean, a1 = v[h][i].y - mean, a2 = v[h][i].z - mean, a3 = v[h][i].w - mean;
        q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
      }
      const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)K + xs.eps);
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        v[h][i].x = (v[h][i].x - mean) * rstd * g[i].x + be[i].x; v[h][i].y = (v[h][i].y - mean) * rstd * g[i].y + be[i].y;
        v[h][i].z = (v[h][i].z - mean) * rstd * g[i].z + be[i].z; v[h][i].w = (v[h][i].w - mean) * rstd * g[i].w + be[i].w;
      }
    }
  }
}

// Fill Xs[BT][K] (f32) for batch rows b0..b0+BT-1.
__device__ __forceinline__ void load_x_tile(const XSrc& xs, float* Xs, int b0, int B, int K, bool publish) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < BT; r += LIN_WARPS) {
    const int b = b0 + r;
    float* row = Xs + (size_t)r * K;
    if (b >= B) { for (int c = lane; c < K; c += 32) row[c] = 0.f; continue; }
    if (xs.mode == XMODE_PLAIN) {
      const float* src = xs.x + (int64_t)b * xs.ldx;
      for (int c = lane * 4; c < K; c += 128) *reinterpret_cast<float4*>(row + c) = *reinterpret_cast<const float4*>(src + c);
    } else {
      operand_row<false>(xs, b, K, row);
    }
    if (publish && xs.xn_out) {
      __syncwarp();
      for (int c = lane; c < K; c += 32) xs.xn_out[(int64_t)b * K + c] = row[c];
    }
  }
}

// Compile-time-K operand tile: every global load of the tile is in flight before the first use.
//   PLAIN      : cp.async 16-byte chunks straight into shared memory; the only form of an operand wider than a model row
//                (FFN2, K = 2048: mdc_model_create caps the model width at MDC_MAX_DEC_DIM)
//   LN / EMBED : a warp owns rows (warp, warp+8), built in lockstep (operand_rows_vec)
template <int K>
__device__ __forceinline__ void load_x_tile_fast(const XSrc& xs, float* Xs, int b0, int B, bool publish) {
  static_assert(K % 128 == 0, "K must be a multiple of 128");
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (K > MDC_MAX_DEC_DIM || xs.mode == XMODE_PLAIN) {
    constexpr int CH = K / 4;   // 16-byte chunks per row
#pragma unroll 8
    for (int i = threadIdx.x; i < BT * CH; i += LIN_THREADS) {
      const int r = i / CH, c4 = i - r * CH, b = b0 + r;
      if (b < B) cp_async16(smem_u32(Xs + (size_t)r * K + c4 * 4), xs.x + (int64_t)b * xs.ldx + c4 * 4);
      else *reinterpret_cast<float4*>(Xs + (size_t)r * K + c4 * 4) = make_float4(0, 0, 0, 0);
    }
    cp_async_wait_all();
    if (publish && xs.xn_out) {
      __syncthreads();
      for (int i = threadIdx.x; i < BT * CH; i += LIN_THREADS) {
        const int r = i / CH, c4 = i - r * CH, b = b0 + r;
        if (b < B) *reinterpret_cast<float4*>(xs.xn_out + (int64_t)b * K + c4 * 4) = *reinterpret_cast<const float4*>(Xs + (size_t)r * K + c4 * 4);
      }
    }
    return;
  }
  if constexpr (K <= MDC_MAX_DEC_DIM) {
    constexpr int NV = K / 128;
    float4 v[2][NV];
    operand_rows_vec<NV, 2>(xs, b0 + warp, B, v);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = warp + 8 * h, b = b0 + r;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        *reinterpret_cast<float4*>(Xs + (size_t)r * K + (i * 32 + lane) * 4) = (b < B) ? v[h][i] : make_float4(0, 0, 0, 0);
        if (publish && xs.xn_out && b < B) *reinterpret_cast<float4*>(xs.xn_out + (int64_t)b * K + (i * 32 + lane) * 4) = v[h][i];
      }
    }
  }
}

// raw 8-element weight slice held in registers until the operand tile is ready
template <typename T> struct Raw8;
template <> struct Raw8<bf16> {
  uint4 v;
  __device__ __forceinline__ void load(const bf16* p) { v = __ldg(reinterpret_cast<const uint4*>(p)); }
  __device__ __forceinline__ void zero() { v = make_uint4(0, 0, 0, 0); }
  __device__ __forceinline__ void unpack(float* f) const {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 t = __bfloat1622float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
  }
};
template <> struct Raw8<__half> {      // decode-loop weights under bf16 precision
  uint4 v;
  __device__ __forceinline__ void load(const __half* p) { v = __ldg(reinterpret_cast<const uint4*>(p)); }
  __device__ __forceinline__ void zero() { v = make_uint4(0, 0, 0, 0); }
  __device__ __forceinline__ void unpack(float* f) const {
    const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 t = __half22float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
  }
};
template <> struct Raw8<float> {
  float4 a, b;
  __device__ __forceinline__ void load(const float* p) { a = __ldg(reinterpret_cast<const float4*>(p)); b = __ldg(reinterpret_cast<const float4*>(p + 4)); }
  __device__ __forceinline__ void zero() { a = make_float4(0, 0, 0, 0); b = a; }
  __device__ __forceinline__ void unpack(float* f) const { f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w; }
};

// Y[B,N] = act(Xeff[B,K] . W[N,K]^T + bias), K = KCH*256.  grid = (N / (LIN_WARPS*RW), ceil(B/BT)).
// A warp owns RW output columns; lanes split K in 8-element (128-bit) slices.  ALL of the warp's weight
// slices are requested before the operand tile is built, so the weight fetch, the operand fetch and the
// LayerNorm-on-load overlap instead of forming a chain of dependent round trips.
template <typename TW, int RW, int KCH, bool RELU>
__global__ void __launch_bounds__(LIN_THREADS) dec_linear_kernel(XSrc xs, const TW* __restrict__ W, const float* __restrict__ bias,
                                                                  float* __restrict__ Y, int64_t ldy, int B, int N) {
  if (batch_done(xs.done)) return;
  constexpr int K = KCH * 256;
  extern __shared__ __align__(16) float Xs[];
  const int b0 = blockIdx.y * BT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = (blockIdx.x * LIN_WARPS + warp) * RW;
  Raw8<TW> w[RW][KCH];
#pragma unroll
  for (int c = 0; c < RW; ++c)
#pragma unroll
    for (int kc = 0; kc < KCH; ++kc) {
      if (n0 + c < N) w[c][kc].load(W + (int64_t)(n0 + c) * K + kc * 256 + lane * 8);
      else w[c][kc].zero();
    }
  load_x_tile_fast<K>(xs, Xs, b0, B, blockIdx.x == 0);
  __syncthreads();
  float acc[RW][BT];
#pragma unroll
  for (int c = 0; c < RW; ++c)
#pragma unroll
    for (int r = 0; r < BT; ++r) acc[c][r] = 0.f;
#pragma unroll
  for (int kc = 0; kc < KCH; ++kc) {
    float wf[RW][8];
#pragma unroll
    for (int c = 0; c < RW; ++c) w[c][kc].unpack(wf[c]);
    const float* xp = Xs + kc * 256 + lane * 8;
#pragma unroll
    for (int r = 0; r < BT; ++r) {
      float4 xa = *reinterpret_cast<const float4*>(xp + (size_t)r * K);
      float4 xb = *reinterpret_cast<const float4*>(xp + (size_t)r * K + 4);
#pragma unroll
      for (int c = 0; c < RW; ++c) {
        float a = acc[c][r];
        a = fmaf(wf[c][0], xa.x, a); a = fmaf(wf[c][1], xa.y, a); a = fmaf(wf[c][2], xa.z, a); a = fmaf(wf[c][3], xa.w, a);
        a = fmaf(wf[c][4], xb.x, a); a = fmaf(wf[c][5], xb.y, a); a = fmaf(wf[c][6], xb.z, a); a = fmaf(wf[c][7], xb.w, a);
        acc[c][r] = a;
      }
    }
  }
#pragma unroll
  for (int c = 0; c < RW; ++c) {
    const int n = n0 + c;
    const float bv = (n < N && bias) ? bias[n] : 0.f;
#pragma unroll
    for (int r = 0; r < BT; ++r) {
      float v = warp_sum(acc[c][r]);
      if (lane == r && n < N && b0 + r < B) {
        v += bv;
        if (RELU) v = fmaxf(v, 0.f);
        Y[(int64_t)(b0 + r) * ldy + n] = v;
      }
    }
  }
}

// generic-K variant (K % 8 == 0 only; e.g. the 64-wide tiny configuration)
template <typename TW, bool RELU>
__global__ void __launch_bounds__(LIN_THREADS) dec_linear_generic_kernel(XSrc xs, const TW* __restrict__ W, const float* __restrict__ bias,
                                                                          float* __restrict__ Y, int64_t ldy, int B, int N, int K) {
  if (batch_done(xs.done)) return;
  extern __shared__ __align__(16) float Xs[];
  const int b0 = blockIdx.y * BT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.x * LIN_WARPS + warp;
  load_x_tile(xs, Xs, b0, B, K, blockIdx.x == 0);
  __syncthreads();
  float acc[BT];
#pragma unroll
  for (int r = 0; r < BT; ++r) acc[r] = 0.f;
  for (int k0 = lane * 8; k0 < K; k0 += 256) {
    float w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (n < N) load8(W + (int64_t)n * K + k0, w);
#pragma unroll
    for (int r = 0; r < BT; ++r) {
      float4 xa = *reinterpret_cast<const float4*>(Xs + (size_t)r * K + k0);
      float4 xb = *reinterpret_cast<const float4*>(Xs + (size_t)r * K + k0 + 4);
      float a = acc[r];
      a = fmaf(w[0], xa.x, a); a = fmaf(w[1], xa.y, a); a = fmaf(w[2], xa.z, a); a = fmaf(w[3], xa.w, a);
      a = fmaf(w[4], xb.x, a); a = fmaf(w[5], xb.y, a); a = fmaf(w[6], xb.z, a); a = fmaf(w[7], xb.w, a);
      acc[r] = a;
    }
  }
  const float bv = (n < N && bias) ? bias[n] : 0.f;
#pragma unroll
  for (int r = 0; r < BT; ++r) {
    float v = warp_sum(acc[r]);
    if (lane == r && n < N && b0 + r < B) {
      v += bv;
      if (RELU) v = fmaxf(v, 0.f);
      Y[(int64_t)(b0 + r) * ldy + n] = v;
    }
  }
}

// ---- tensor-core form of the same linear for batches of 16 and more (fp16 decode-loop weights) ----------------------------------
// Y[B,N] = act(Xeff[B,K] . W[N,K]^T + bias) with the WEIGHT rows as the M operand of mma.sync.m16n8k16 and the images as N = 8
// column blocks, like the fused cluster kernel's projections: a CTA of 8 warps owns 64 weight rows (4 row groups of 16) x 64 images
// (2 halves of 4 column blocks); every weight is read from global memory ONCE per 64 images (the FFMA kernel above re-streams the
// weights per 16 images and does the arithmetic on the FP32 pipe: 2.6 ms per token-step at dim 1024 / 8 layers / B = 64).
// The operand rows (plain / LayerNorm-on-load / embedding, the same three sources) are built once per CTA as IEEE half in shared
// memory (the precision policy of the fused kernel: fp16 projection operands).  Weight fragments come straight from global memory:
// lane (g, q) loads the 16 bytes W[row g (+8)][32 kb + 8 q .. +8) and uses them as the A fragments of two k-steps under the k
// permutation logical (step s, 2q + j, +8 hi) <-> physical 8 q + 4 s + 2 hi + j, which the B fragment (one 8-byte shared load
// X[image][32 kb + 8 q + 4 s .. +4)) follows -- a dot product does not care in which order k is enumerated.
constexpr int MMA_ROWS = 64;       // weight rows per CTA
constexpr int MMA_IMGS = 64;       // images per CTA
constexpr int MMA_KC = 1024;       // operand columns held in shared memory at a time
constexpr int MMA_PAD = 4;         // halves of row padding: row pitch = 2 words mod 32 (two-way conflicts at worst on the 8-byte loads)

// LayerNorm-on-load / embedding operand rows, built ONCE per linear (one warp per image, all images in parallel) as IEEE half in
// global memory, and published as the next residual (xn_out, f32).  Building them inside every CTA of the linear -- eight rows per
// warp, one after the other, three dependent memory round trips each -- was 75 % of that kernel's time (ncu, profiles/r2w).
// K % 128 == 0 (every model width on the path): 128-bit loads and stores -- the scalar form below issues 128 loads and 64 stores per
// lane for a 1024-wide row and was LSU-latency bound (7.9 us per launch at B = 64, a quarter of a dim-1024 token-step)
template <int NV>
__global__ void __launch_bounds__(LIN_THREADS) prep_x_half_vec_kernel(XSrc xs, __half* __restrict__ xh, int B) {
  if (batch_done(xs.done)) return;
  constexpr int K = NV * 128;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * LIN_WARPS + warp;
  if (b >= B) return;
  float4 v[1][NV];
  operand_rows_vec<NV, 1>(xs, b, B, v);
  uint2* oh = reinterpret_cast<uint2*>(xh + (int64_t)b * K) + lane;
  float4* of = xs.xn_out ? reinterpret_cast<float4*>(xs.xn_out + (int64_t)b * K) + lane : nullptr;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    oh[32 * i] = make_uint2(pack_f16x2_sat(v[0][i].x, v[0][i].y), pack_f16x2_sat(v[0][i].z, v[0][i].w));
    if (of) of[32 * i] = v[0][i];
  }
}

__global__ void __launch_bounds__(LIN_THREADS) prep_x_half_kernel(XSrc xs, __half* __restrict__ xh, int B, int K) {
  if (batch_done(xs.done)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * LIN_WARPS + warp;
  if (b >= B) return;
  float v[MDC_MAX_DEC_DIM / 32];
  operand_row<true>(xs, b, K, v);
#pragma unroll
  for (int i = 0; i < MDC_MAX_DEC_DIM / 32; ++i) {
    const int c = lane + 32 * i;
    if (c < K) {
      xh[(int64_t)b * K + c] = f16_sat(v[i]);
      if (xs.xn_out) xs.xn_out[(int64_t)b * K + c] = v[i];
    }
  }
}

// operand rows b0 .. b0+63, columns [k0, k0+kc) -> Xh[64][kc + MMA_PAD] (fp16); rows >= B are zero.
//   HALF : rows already in IEEE half (prep_x_half_kernel): 8-byte cp.async chunks, every row in flight at once
//   PLAIN: f32 rows (attention outputs, the FFN hidden), converted on the way; two rows per warp in flight
__device__ __forceinline__ void build_x_half(const XSrc& xs, __half* Xh, int b0, int B, int K, int k0, int kc, bool publish) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pitch = kc + MMA_PAD;
  if (xs.mode == XMODE_HALF) {
    for (int r = warp; r < MMA_IMGS; r += LIN_WARPS) {          // a warp copies whole rows: 8-byte chunks, 256 bytes per instruction
      const int b = b0 + r;
      __half* dst = Xh + (size_t)r * pitch;
      const __half* src = xs.xh + (int64_t)min(b, B - 1) * K + k0;
      if (b < B) { for (int c = lane * 4; c < kc; c += 128) cp_async8(smem_u32(dst + c), src + c); }
      else { for (int c = lane * 4; c < kc; c += 128) *reinterpret_cast<uint2*>(dst + c) = make_uint2(0u, 0u); }
    }
    cp_async_wait_all();
    return;
  }
  for (int r = warp; r < MMA_IMGS; r += 2 * LIN_WARPS) {      // rows r and r + 8
    float4 v[2][MMA_KC / 128];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int b = b0 + r + 8 * h;
      const float* src = xs.x + (int64_t)min(b, B - 1) * xs.ldx + k0;
#pragma unroll
      for (int i = 0; i < MMA_KC / 128; ++i) { const int c = lane * 4 + 128 * i; if (c < kc) v[h][i] = *reinterpret_cast<const float4*>(src + c); }
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int b = b0 + r + 8 * h;
      __half* row = Xh + (size_t)(r + 8 * h) * pitch;
#pragma unroll
      for (int i = 0; i < MMA_KC / 128; ++i) {
        const int c = lane * 4 + 128 * i;
        if (c < kc) {
          *reinterpret_cast<uint2*>(row + c) = b < B ? make_uint2(pack_f16x2_sat(v[h][i].x, v[h][i].y), pack_f16x2_sat(v[h][i].z, v[h][i].w)) : make_uint2(0u, 0u);
          if (publish && xs.xn_out && b < B) *reinterpret_cast<float4*>(xs.xn_out + (int64_t)b * K + k0 + c) = v[h][i];
        }
      }
    }
  }
}

template <bool RELU>
__global__ void __launch_bounds__(LIN_THREADS) dec_linear_mma_kernel(XSrc xs, const __half* __restrict__ W, const float* __restrict__ bias,
                                                                      float* __restrict__ Y, int64_t ldy, int B, int N, int K) {
  if (batch_done(xs.done)) return;
  extern __shared__ __align__(16) uint8_t mma_smem[];
  __half* Xh = reinterpret_cast<__half*>(mma_smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  const int b0 = blockIdx.y * MMA_IMGS;
  const int r0 = blockIdx.x * MMA_ROWS + (warp & 3) * 16;           // this warp's 16 weight rows
  const int nb0 = (warp >> 2) * 4;                                  // this warp's four 8-image column blocks
  const int row_a = min(r0 + g, N - 1), row_b = min(r0 + g + 8, N - 1);   // rows past N are computed on a valid row and never stored
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }
  for (int k0 = 0; k0 < K; k0 += MMA_KC) {
    const int kc = min(MMA_KC, K - k0), pitch = kc + MMA_PAD;
    if (k0) __syncthreads();
    build_x_half(xs, Xh, b0, B, K, k0, kc, blockIdx.x == 0);
    __syncthreads();
    const __half* wa = W + (int64_t)row_a * K + k0 + 8 * q;
    const __half* wb = W + (int64_t)row_b * K + k0 + 8 * q;
    const __half* xb = Xh + (size_t)(8 * nb0 + g) * pitch + 8 * q;
    const int nkb = kc >> 5;
    constexpr int PF = 8;                                           // weight slices of eight 32-column blocks in flight per lane
    uint4 alo[PF], ahi[PF];
#pragma unroll
    for (int i = 0; i < PF; ++i)
      if (i < nkb) { alo[i] = __ldg(reinterpret_cast<const uint4*>(wa + 32 * i)); ahi[i] = __ldg(reinterpret_cast<const uint4*>(wb + 32 * i)); }
    for (int kb0 = 0; kb0 < nkb; kb0 += PF) {
#pragma unroll
      for (int i = 0; i < PF; ++i) {
        const int kb = kb0 + i;
        if (kb < nkb) {
          const uint4 lo = alo[i], hi = ahi[i];
          if (kb + PF < nkb) { alo[i] = __ldg(reinterpret_cast<const uint4*>(wa + 32 * (kb + PF))); ahi[i] = __ldg(reinterpret_cast<const uint4*>(wb + 32 * (kb + PF))); }
#pragma unroll
          for (int nb = 0; nb < 4; ++nb) {
            const uint2 x0 = *reinterpret_cast<const uint2*>(xb + (size_t)(8 * nb) * pitch + 32 * kb);
            const uint2 x1 = *reinterpret_cast<const uint2*>(xb + (size_t)(8 * nb) * pitch + 32 * kb + 4);
            const uint32_t a0[4] = {lo.x, hi.x, lo.y, hi.y}, a1[4] = {lo.z, hi.z, lo.w, hi.w};
            mma_m16n8k16<__half>(acc[nb], a0, x0.x, x0.y);
            mma_m16n8k16<__half>(acc[nb], a1, x1.x, x1.y);
          }
        }
      }
    }
  }
  // acc[nb][e]: row r0 + g + 8 (e >> 1), image 8 (nb0 + nb) + 2 q + (e & 1)
#pragma unroll
  for (int e2 = 0; e2 < 2; ++e2) {
    const int n = r0 + g + 8 * e2;
    if (n < N) {
      const float bv = bias ? bias[n] : 0.f;
#pragma unroll
      for (int nb = 0; nb < 4; ++nb)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int b = b0 + 8 * (nb0 + nb) + 2 * q + j;
          if (b < B) {
            float v = acc[nb][2 * e2 + j] + bv;
            if (RELU) v = fmaxf(v, 0.f);
            Y[(int64_t)b * ldy + n] = v;
          }
        }
    }
  }
}

// ---- weight-streaming form of the tensor-core linear (wide geometries: dim 1024 / 8 layers, trail_01.py:158-160) ----------------
// dec_linear_mma_kernel gives a CTA 64 weight rows: N = 1024 is 16 CTAs, each pulling 128 KB of weights through eight loads per lane
// after it has staged all 64 operand rows in shared memory -- 16 of 148 SMs stream the weights (25-36 us per linear, 72 GB/s in ncu,
// profiles/r2y).  Here a CTA owns only 16 weight rows (one MMA row tile) and its eight warps split K: warp w takes the 32-column
// blocks w, w+8, ... of those rows for all 64 images, so N = 1024 is 64 CTAs, every weight byte of the linear is requested in the
// first few hundred cycles of the launch (32-64 KB in flight per CTA), nothing waits for a staged operand tile, and there is no
// barrier before the cross-warp sum.  Operand rows are IEEE half in global memory (L2-resident: B x K halves, written by
// prep_x_half_kernel, by the attention kernels or by the previous linear of this kind) and are loaded straight into the B fragments:
// lane (g, q) reads the 16 bytes X[image 8 nb + g][32 kb + 8 q .. +8) = both k-steps of the block under the same k permutation as
// above.  The eight K-partials of the 16 x 64 tile are summed through shared memory in warp order (deterministic, batch-invariant).
constexpr int STREAM_ROWS = 16;
constexpr int STREAM_MT2_MIN_N = 2048;       // linears at least this wide take two 16-row tiles per CTA (A/B on B200, B = 64: every linear:
                                             // serial token-step +10 %, pipeline +9 %; N >= 2048 only: serial -0.5 %, pipeline +5 %)
constexpr int STREAM_PITCH = MMA_IMGS + 8;   // floats per row of a warp's partial tile
constexpr int STREAM_SLOTS = 4;              // 32-column operand blocks in flight per warp (K = 1024: the warp's whole share)
constexpr int STREAM_SLOT_BYTES = MMA_IMGS * 64;                                   // [64 images][32 halves]
constexpr int STREAM_SMEM = LIN_WARPS * STREAM_SLOTS * STREAM_SLOT_BYTES;          // 128 KB; the partial tiles alias it afterwards

// MT = 16-row tiles per CTA.  Two tiles share every operand fragment read and halve the CTA count: the same kernel latency for half the SM
// residency, which is what the batch pipeline (several batches' chains side by side, one such CTA per SM) is bound by.
template <bool RELU, int MT>
__global__ void __launch_bounds__(LIN_THREADS) dec_linear_stream_kernel(const __half* __restrict__ X, int64_t ldx, const __half* __restrict__ W,
                                                                         const float* __restrict__ bias, float* __restrict__ Y, int64_t ldy,
                                                                         __half* __restrict__ Yh, int64_t ldyh, int B, int N, int K,
                                                                         const uint8_t* __restrict__ pf, int pf_lines, const int* done) {
  if (batch_done(done)) return;
  constexpr int ROWS = STREAM_ROWS * MT;
  static_assert(LIN_WARPS * ROWS * STREAM_PITCH * 4 <= STREAM_SMEM, "partial tiles must fit into the operand ring");
  extern __shared__ __align__(128) uint8_t stream_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  const int b0 = blockIdx.y * MMA_IMGS, r0 = blockIdx.x * ROWS;
  const __half* wa[MT]; const __half* wb[MT];                               // rows past N: computed on a valid row, never stored
#pragma unroll
  for (int m = 0; m < MT; ++m) {
    wa[m] = W + (int64_t)min(r0 + 16 * m + g, N - 1) * K + 32 * warp + 8 * q;      // block i of this warp: + 256 i
    wb[m] = W + (int64_t)min(r0 + 16 * m + g + 8, N - 1) * K + 32 * warp + 8 * q;
  }
  const int nkb = K >> 8;                                                   // 32-column blocks per warp (K % 256 == 0)
  constexpr int PF = 8 / MT;
  uint4 alo[MT][PF], ahi[MT][PF];
#pragma unroll
  for (int i = 0; i < PF; ++i)
    if (i < nkb) {
#pragma unroll
      for (int m = 0; m < MT; ++m) { alo[m][i] = __ldg(reinterpret_cast<const uint4*>(wa[m] + 256 * i)); ahi[m][i] = __ldg(reinterpret_cast<const uint4*>(wb[m] + 256 * i)); }
    }
  // the NEXT linear's weights (168 MB of decode-loop weights per token-step do not stay in the 126 MB L2) are pulled into L2 while this
  // linear and the one or two small kernels behind it run: its weight requests then cost an L2 round trip instead of an HBM one
  if (pf != nullptr && blockIdx.y == 0)
    for (int i = blockIdx.x * LIN_THREADS + threadIdx.x; i < pf_lines; i += gridDim.x * LIN_THREADS)
      prefetch_l2(pf + (size_t)i * 128);
  // operand ring of this warp: slot = [64 images][4 x 16 bytes]; lane l copies the 16-byte pieces l, l + 32, ... (piece = 4 image + part)
  const uint32_t ring = smem_u32(stream_smem) + warp * (STREAM_SLOTS * STREAM_SLOT_BYTES);
  // image slots past the batch are zeroed once and never copied (clamping them to the last row made thousands of L2 requests hit the
  // same two sectors: a B = 16 step was twice as slow as a B = 64 step)
  const __half* xsrc[8];
  uint32_t live = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int piece = lane + 32 * j, img = piece >> 2, part = piece & 3;
    xsrc[j] = X + (int64_t)min(b0 + img, B - 1) * ldx + 32 * warp + 8 * part;
    if (b0 + img < B) live |= 1u << j;
    else {
#pragma unroll
      for (int sl = 0; sl < STREAM_SLOTS; ++sl)
        sts128(ring + sl * STREAM_SLOT_BYTES + piece * 16, 0u, 0u, 0u, 0u);
    }
  }
  auto fetch = [&](int it) {
    if (it < nkb) {
      const uint32_t dst = ring + (it % STREAM_SLOTS) * STREAM_SLOT_BYTES + lane * 16;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (live >> j & 1) cp_async16(dst + 512 * j, xsrc[j] + 256 * it);
    }
    cp_async_commit();                                                      // one group per block, empty past the end
  };
#pragma unroll
  for (int i = 0; i < STREAM_SLOTS; ++i) fetch(i);
  float acc[MT][8][4];
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) { acc[m][nb][0] = acc[m][nb][1] = acc[m][nb][2] = acc[m][nb][3] = 0.f; }
  for (int i0 = 0; i0 < nkb; i0 += PF) {
#pragma unroll
    for (int i = 0; i < PF; ++i) {
      const int it = i0 + i;
      if (it < nkb) {
        uint4 lo[MT], hi[MT];
#pragma unroll
        for (int m = 0; m < MT; ++m) {
          lo[m] = alo[m][i]; hi[m] = ahi[m][i];
          if (it + PF < nkb) { alo[m][i] = __ldg(reinterpret_cast<const uint4*>(wa[m] + 256 * (it + PF))); ahi[m][i] = __ldg(reinterpret_cast<const uint4*>(wb[m] + 256 * (it + PF))); }
        }
        cp_async_wait<STREAM_SLOTS - 1>();
        __syncwarp();
        const uint32_t src = ring + (it % STREAM_SLOTS) * STREAM_SLOT_BYTES + g * 64 + q * 16;
#pragma unroll
        for (int nb = 0; nb < 8; ++nb) {
          const uint4 xv = lds128(src + 512 * nb);
#pragma unroll
          for (int m = 0; m < MT; ++m) {
            const uint32_t a0[4] = {lo[m].x, hi[m].x, lo[m].y, hi[m].y}, a1[4] = {lo[m].z, hi[m].z, lo[m].w, hi[m].w};
            mma_m16n8k16<__half>(acc[m][nb], a0, xv.x, xv.y);
            mma_m16n8k16<__half>(acc[m][nb], a1, xv.z, xv.w);
          }
        }
        __syncwarp();
        fetch(it + STREAM_SLOTS);
      }
    }
  }
  cp_async_wait<0>();
  __syncthreads();                                                          // every warp is done with its ring: the partial tiles alias it
  float (*red)[ROWS][STREAM_PITCH] = reinterpret_cast<float (*)[ROWS][STREAM_PITCH]>(stream_smem);
  // acc[m][nb][e]: row 16 m + g + 8 (e >> 1), image 8 nb + 2 q + (e & 1)
#pragma unroll
  for (int m = 0; m < MT; ++m)
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
      *reinterpret_cast<float2*>(&red[warp][16 * m + g][8 * nb + 2 * q]) = make_float2(acc[m][nb][0], acc[m][nb][1]);
      *reinterpret_cast<float2*>(&red[warp][16 * m + g + 8][8 * nb + 2 * q]) = make_float2(acc[m][nb][2], acc[m][nb][3]);
    }
  __syncthreads();
  const int row = threadIdx.x & (ROWS - 1), n = r0 + row;
  if (n < N) {
    const float bv = bias ? bias[n] : 0.f;
    constexpr int IPP = LIN_THREADS / ROWS;                                 // images per pass
#pragma unroll
    for (int j = 0; j < MMA_IMGS / IPP; ++j) {
      const int img = (threadIdx.x / ROWS) + IPP * j, b = b0 + img;
      if (b < B) {
        float v = red[0][row][img];
#pragma unroll
        for (int w = 1; w < LIN_WARPS; ++w) v += red[w][row][img];
        v += bv;
        if (RELU) v = fmaxf(v, 0.f);
        if (Y) Y[(int64_t)b * ldy + n] = v;
        if (Yh) Yh[(int64_t)b * ldyh + n] = f16_sat(v);
      }
    }
  }
}

// ---- attention of ONE query per (image, head) over a key/value set ---------------------------------
// warp == head.  A key's HD channels are split over LPK = HD/8 lanes (one 128-bit load each), so a warp
// covers 32/LPK keys per pass with fully-used sectors; passes are unrolled x4 with the loads issued first
// (memory-level parallelism instead of a chain of dependent round trips).  Softmax max/sum are warp
// shuffles; P.V uses the same (key slot, 8-channel chunk) lane mapping.
template <typename TKV, int HD, typename KeyPtr, typename Bias>
__device__ __forceinline__ void attend_one(const float* q /*smem, HD, pre-scaled*/, float* sc /*smem, nkeys*/, int nkeys,
                                           KeyPtr kv_ptr, Bias bias, float* out /*HD*/, __half* outh = nullptr /*HD, IEEE-half twin*/) {
  constexpr int LPK = HD / 8, KPI = 32 / LPK, UN = 4;
  const int lane = threadIdx.x & 31, sub = lane % LPK, kslot = lane / LPK;
  float qv[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) qv[j] = q[sub * 8 + j];
  float mx = -INFINITY;
  for (int u0 = 0; u0 < nkeys; u0 += KPI * UN) {
    Raw8<TKV> r[UN];
#pragma unroll
    for (int i = 0; i < UN; ++i) {
      const int u = u0 + i * KPI + kslot;
      if (u < nkeys) r[i].load(kv_ptr(u, 0, sub)); else r[i].zero();
    }
#pragma unroll
    for (int i = 0; i < UN; ++i) {
      const int u = u0 + i * KPI + kslot;
      float kf[8]; r[i].unpack(kf);
      float sdot = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) sdot = fmaf(qv[j], kf[j], sdot);
#pragma unroll
      for (int o = 1; o < LPK; o <<= 1) sdot += __shfl_xor_sync(0xffffffffu, sdot, o);
      if (u < nkeys) {
        sdot += bias(u);
        if (sub == 0) sc[u] = sdot;
        mx = fmaxf(mx, sdot);
      }
    }
  }
  mx = warp_max(mx);
  __syncwarp();
  float sum = 0.f;
  for (int u = lane; u < nkeys; u += 32) { float e = expf(sc[u] - mx); sc[u] = e; sum += e; }
  sum = warp_sum(sum);
  __syncwarp();
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int u0 = 0; u0 < nkeys; u0 += KPI * UN) {
    Raw8<TKV> r[UN];
#pragma unroll
    for (int i = 0; i < UN; ++i) {
      const int u = u0 + i * KPI + kslot;
      if (u < nkeys) r[i].load(kv_ptr(u, 1, sub)); else r[i].zero();
    }
#pragma unroll
    for (int i = 0; i < UN; ++i) {
      const int u = u0 + i * KPI + kslot;
      const float p = (u < nkeys) ? sc[u] : 0.f;
      float vf[8]; r[i].unpack(vf);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(p, vf[j], acc[j]);
    }
  }
#pragma unroll
  for (int o = LPK; o < 32; o <<= 1) {
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], o);
  }
  if (kslot == 0) {
    const float inv = 1.0f / sum;
#pragma unroll
    for (int j = 0; j < 8; ++j) out[sub * 8 + j] = acc[j] * inv;
    if (outh) {
#pragma unroll
      for (int j = 0; j < 8; ++j) outh[sub * 8 + j] = f16_sat(acc[j] * inv);
    }
  }
  __syncwarp();
}

// self-attention: appends this step's k,v to the paged cache, then attends over slots 0..t.
// pool layout: [page][layer][head][k|v][page_tokens][hd] -- the K and V rows of one (page, layer, head) are one contiguous
// 2 * page_tokens * hd block (the fused decode kernel fetches it with ONE bulk copy).  When a row is 64 bytes (hd = 32, 16-bit
// cache) the 16-byte chunk c of token r is stored at chunk c ^ ((r >> 1) & 3): the bank-conflict-free pattern of the fused kernel's
// ldmatrix reads (what TMA SWIZZLE_64B would produce), shared by both implementations.
template <typename TKV, int HD>
__device__ __forceinline__ int kv_chunk(int r, int c) { return (HD * (int)sizeof(TKV) == 64) ? (c ^ ((r >> 1) & 3)) : c; }

template <typename TKV, int HD>
__global__ void dec_self_attn_kernel(const float* __restrict__ qkv /*[B,3d]*/, TKV* __restrict__ pool,
                                     const int32_t* __restrict__ page_table, int pages_per_seq, int PT, int n_layers, int layer,
                                     const int32_t* __restrict__ tokens, int tokens_ld, int pad_idx, int t, int d,
                                     float scale, float* __restrict__ o /*[B,d]*/, __half* __restrict__ oh /*[B,d] or NULL*/, const int* done) {
  if (batch_done(done)) return;
  constexpr int hd = HD;
  extern __shared__ float sm[];
  const int b = blockIdx.x, head = threadIdx.x >> 5, lane = threadIdx.x & 31, heads = blockDim.x >> 5;
  float* q = sm + head * hd;
  float* sc = sm + heads * hd + head * (t + 1);
  int* pt = reinterpret_cast<int*>(sm + heads * (hd + t + 1)) + head * pages_per_seq;   // per-warp copy of the page ids: one round trip
  const float* row = qkv + (int64_t)b * 3 * d;
  for (int j = lane; j <= t / PT; j += 32) pt[j] = page_table[(int64_t)b * pages_per_seq + j];
  __syncwarp();
  const int64_t plane = (int64_t)PT * hd;                   // the k or v rows of one (page, layer, head)
  auto kv_base = [&](int u, int which) -> TKV* {
    return pool + ((((int64_t)pt[u / PT] * n_layers + layer) * heads + head) * 2 + which) * plane + (int64_t)(u % PT) * hd;
  };
  {  // append k_t, v_t (this head's channels) and stage q
    TKV* kdst = kv_base(t, 0); TKV* vdst = kv_base(t, 1);
    const int r = t % PT;
    for (int c = lane; c < hd; c += 32) {
      q[c] = row[head * hd + c] * scale;
      const int pc = kv_chunk<TKV, HD>(r, c >> 3) * 8 + (c & 7);
      kdst[pc] = from_f<TKV>(row[d + head * hd + c]);
      vdst[pc] = from_f<TKV>(row[2 * d + head * hd + c]);
    }
  }
  __syncwarp();
  auto kv_ptr = [&](int u, int which, int sub) -> const TKV* { return kv_base(u, which) + kv_chunk<TKV, HD>(u % PT, sub) * 8; };
  auto bias = [&](int u) -> float { return tokens[(int64_t)b * tokens_ld + u] == pad_idx ? 1.0f : 0.0f; };
  attend_one<TKV, HD>(q, sc, t + 1, kv_ptr, bias, o + (int64_t)b * d + head * hd, oh ? oh + (int64_t)b * d + head * hd : nullptr);
}

// cross-attention over the S memory keys of image b; cross_kv layer plane: [B*S][2d] (K | V)
template <typename TKV, int HD>
__global__ void dec_cross_attn_kernel(const float* __restrict__ qc /*[B,d]*/, const TKV* __restrict__ ckv_layer, int S, int d,
                                      float scale, float* __restrict__ o, const int* done) {
  if (batch_done(done)) return;
  constexpr int hd = HD;
  extern __shared__ float sm[];
  const int b = blockIdx.x, head = threadIdx.x >> 5, lane = threadIdx.x & 31, heads = blockDim.x >> 5;
  float* q = sm + head * hd;
  float* sc = sm + heads * hd + head * S;
  for (int c = lane; c < hd; c += 32) q[c] = qc[(int64_t)b * d + head * hd + c] * scale;
  __syncwarp();
  const TKV* base = ckv_layer + (int64_t)b * S * 2 * d + head * hd;
  auto kv_ptr = [&](int u, int which, int sub) -> const TKV* { return base + (int64_t)u * 2 * d + which * d + sub * 8; };
  auto bias = [&](int) -> float { return 0.f; };
  attend_one<TKV, HD>(q, sc, S, kv_ptr, bias, o + (int64_t)b * d + head * hd);
}

// cross-attention of ONE query per (image, head) with the memory keys split over the eight warps of a CTA (grid = heads x B).
// dec_cross_attn_kernel walks the keys of a head with one warp: at head width 128 that is two keys per pass, 98 dependent round
// trips of 2 KB each for S = 196 (45 us per layer at B = 64, 1.1 TB/s).  Here warp w takes the passes w, w + 8, ..., all 512 CTAs of
// a B = 64 launch are resident and every K (then V) byte of the layer is requested within four rounds.  Scores go through shared
// memory; max / sum / the eight partial outputs are combined in warp order (deterministic).  Output as IEEE half = the operand of
// the out-projection.
template <typename TKV, int HD>
__global__ void __launch_bounds__(LIN_THREADS) dec_cross_attn_split_kernel(const float* __restrict__ qc /*[B,d]*/, const TKV* __restrict__ ckv_layer,
                                                                            int S, int d, float scale, __half* __restrict__ oh, const int* done) {
  if (batch_done(done)) return;
  constexpr int LPK = HD / 8, KPI = 32 / LPK, UN = 4;
  extern __shared__ float sm[];
  float* qs = sm;                       // HD
  float* part = qs + HD;                // LIN_WARPS x HD
  float* wred = part + LIN_WARPS * HD;  // 2 x LIN_WARPS
  float* sc = wred + 2 * LIN_WARPS;     // S
  const int head = blockIdx.x, b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, sub = lane % LPK, kslot = lane / LPK;
  const TKV* base = ckv_layer + (int64_t)b * S * 2 * d + head * HD + sub * 8;
  constexpr int STEP = LIN_WARPS * KPI;                 // keys per CTA pass
  const int ufirst = warp * KPI + kslot;
  Raw8<TKV> r[UN], rn[UN];
#pragma unroll
  for (int i = 0; i < UN; ++i) { const int u = ufirst + i * STEP; if (u < S) r[i].load(base + (int64_t)u * 2 * d); else r[i].zero(); }
  for (int c = threadIdx.x; c < HD; c += LIN_THREADS) qs[c] = qc[(int64_t)b * d + head * HD + c] * scale;
  __syncthreads();
  float qv[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) qv[j] = qs[sub * 8 + j];
  float mx = -INFINITY;
  for (int u0 = ufirst; u0 < S; u0 += STEP * UN) {
    const int un = u0 + STEP * UN;
    if (un < S) {
#pragma unroll
      for (int i = 0; i < UN; ++i) { const int u = un + i * STEP; if (u < S) rn[i].load(base + (int64_t)u * 2 * d); else rn[i].zero(); }
    }
#pragma unroll
    for (int i = 0; i < UN; ++i) {
      const int u = u0 + i * STEP;
      float kf[8]; r[i].unpack(kf);
      float sdot = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) sdot = fmaf(qv[j], kf[j], sdot);
#pragma unroll
      for (int of = 1; of < LPK; of <<= 1) sdot += __shfl_xor_sync(0xffffffffu, sdot, of);
      if (u < S) { if (sub == 0) sc[u] = sdot; mx = fmaxf(mx, sdot); }
    }
#pragma unroll
    for (int i = 0; i < UN; ++i) r[i] = rn[i];
  }
  // the first round of V slices is requested before the softmax statistics: its round trip overlaps the two barriers and the exponentials
#pragma unroll
  for (int i = 0; i < UN; ++i) { const int u = ufirst + i * STEP; if (u < S) r[i].load(base + (int64_t)u * 2 * d + d); else r[i].zero(); }
  mx = warp_max(mx);
  if (lane == 0) wred[warp] = mx;
  __syncthreads();
  mx = wred[0];
#pragma unroll
  for (int w = 1; w < LIN_WARPS; ++w) mx = fmaxf(mx, wred[w]);
  float sum = 0.f;
  for (int u = threadIdx.x; u < S; u += LIN_THREADS) { const float e = expf(sc[u] - mx); sc[u] = e; sum += e; }
  sum = warp_sum(sum);
  if (lane == 0) wred[LIN_WARPS + warp] = sum;
  __syncthreads();
  float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int u0 = ufirst; u0 < S; u0 += STEP * UN) {
    const int un = u0 + STEP * UN;
    if (un < S) {
#pragma unroll
      for (int i = 0; i < UN; ++i) { const int u = un + i * STEP; if (u < S) rn[i].load(base + (int64_t)u * 2 * d + d); else rn[i].zero(); }
    }
#pragma unroll
    for (int i = 0; i < UN; ++i) {
      const int u = u0 + i * STEP;
      const float p = (u < S) ? sc[u] : 0.f;
      float vf[8]; r[i].unpack(vf);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(p, vf[j], acc[j]);
    }
#pragma unroll
    for (int i = 0; i < UN; ++i) r[i] = rn[i];
  }
#pragma unroll
  for (int of = LPK; of < 32; of <<= 1) {
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], of);
  }
  if (kslot == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) part[warp * HD + sub * 8 + j] = acc[j];
  }
  __syncthreads();
  float tot = wred[LIN_WARPS];
#pragma unroll
  for (int w = 1; w < LIN_WARPS; ++w) tot += wred[LIN_WARPS + w];
  const float inv = 1.0f / tot;
  for (int c = threadIdx.x; c < HD; c += LIN_THREADS) {
    float v = part[c];
#pragma unroll
    for (int w = 1; w < LIN_WARPS; ++w) v += part[w * HD + c];
    v *= inv;
    oh[(int64_t)b * d + head * HD + c] = f16_sat(v);
  }
}

using namespace mdcsel;


// Stop at EOS on the per-operation path (mdc_decode_state.stop_at_eos), in the decode workspace: fin [B] = image b has finished,
// state[0] = number of finished images, state[1] = all finished (the `done` flag every kernel of a step tests at entry).  NULL = off.
struct StopArgs { int* fin; int* state; int eos; };

// Once per mdc_decode_steps call, before the first step (inside a captured graph: at the start of every replay): the token columns
// t_begin+1..t_end become PAD and the conf columns of steps t_begin..t_end-1 zero -- the values of every position after an image's
// EOS, which the select of a step that runs overwrites with the selected token -- and the finished flags and count come from the
// known prefix (an EOS among columns 1..t_begin).  One CTA.
__global__ void __launch_bounds__(SEL_THREADS) dec_stop_init_kernel(int32_t* __restrict__ tokens, int tokens_ld, float* __restrict__ confs,
                                                                     int confs_ld, int B, int t_begin, int t_end, int pad, StopArgs stop) {
  __shared__ int n_fin;
  if (threadIdx.x == 0) n_fin = 0;
  __syncthreads();
  for (int b = threadIdx.x; b < B; b += SEL_THREADS) {
    int f = 0;
    for (int c = 1; c <= t_begin; ++c) f |= tokens[(int64_t)b * tokens_ld + c] == stop.eos;
    stop.fin[b] = f;
    if (f) atomicAdd(&n_fin, 1);
  }
  const int nt = t_end - t_begin;
  for (int64_t i = threadIdx.x; i < (int64_t)B * nt; i += SEL_THREADS)
    tokens[(i / nt) * tokens_ld + t_begin + 1 + i % nt] = pad;
  const int c0 = (t_begin + 3) / 4, nc = (t_end + 3) / 4 - c0;      // conf columns of the steps t % 4 == 0 in [t_begin, t_end)
  if (confs && nc > 0)
    for (int64_t i = threadIdx.x; i < (int64_t)B * nc; i += SEL_THREADS) confs[(i / nc) * confs_ld + c0 + i % nc] = 0.f;
  __syncthreads();
  if (threadIdx.x == 0) { stop.state[0] = n_fin; stop.state[1] = n_fin == B; }
}

// select for the decode loop: reads the step's logits [B,V] (written by the head linear), optionally copies them
// to the caller's logits tensor, then greedy / top-k / top-p select + max-prob.  One CTA per image.
// With stop at EOS an image that has finished is left alone (its columns hold PAD / 0 from dec_stop_init_kernel); an image that
// selects EOS is marked finished and counted, and the count reaching B sets the all-finished flag.  (An image not yet finished keeps
// the count below B during this launch, so the flag cannot change under a CTA that runs.)
__global__ void __launch_bounds__(SEL_THREADS) dec_select_kernel(const float* __restrict__ step_logits, int V, int Vp2, int t,
                                                                  float* __restrict__ logits_out, int64_t logits_img_stride, int logits_row,
                                                                  int32_t* __restrict__ tokens, int tokens_ld, int forced,
                                                                  float* __restrict__ confs, int confs_ld, const float* __restrict__ uniforms,
                                                                  int uniforms_ld, int top_k, float top_p, StopArgs stop) {
  extern __shared__ __align__(16) float sm[];
  float* lg = sm;             // V
  float* srt = lg + V;        // Vp2
  const int b = blockIdx.x;
  if (stop.fin != nullptr && stop.fin[b]) return;
  for (int i = threadIdx.x; i < V; i += SEL_THREADS) {
    float v = step_logits[(int64_t)b * V + i];
    lg[i] = v;
    if (logits_out) logits_out[(int64_t)b * logits_img_stride + (int64_t)logits_row * V + i] = v;
  }
  __syncthreads();
  if (forced && !(confs && (t % 4 == 0))) return;
  const bool sample = (top_k != 0 || top_p != 1.0f) && uniforms != nullptr;
  float u = sample ? uniforms[(int64_t)b * uniforms_ld + t] : 0.f;
  int token; float conf;
  select_from_logits(lg, srt, V, Vp2, top_k, top_p, sample, u, token, conf);
  if (threadIdx.x == 0) {
    if (!forced) tokens[(int64_t)b * tokens_ld + t + 1] = token;
    if (confs && (t % 4 == 0)) confs[(int64_t)b * confs_ld + t / 4] = conf;
    if (stop.fin != nullptr && token == stop.eos) {
      stop.fin[b] = 1;
      if (atomicAdd(&stop.state[0], 1) + 1 == (int)gridDim.x) stop.state[1] = 1;
    }
  }
}

__global__ void __launch_bounds__(SEL_THREADS) select_kernel(const float* __restrict__ logits, int64_t ld, int V, int Vp2, int top_k,
                                                             float top_p, const float* __restrict__ uniforms, int32_t* __restrict__ token_out,
                                                             float* __restrict__ conf_out, float* __restrict__ prob_out) {
  extern __shared__ __align__(16) float sm[];
  float* lg = sm; float* srt = sm + V;
  const int b = blockIdx.x;
  for (int i = threadIdx.x; i < V; i += SEL_THREADS) lg[i] = logits[(int64_t)b * ld + i];
  __syncthreads();
  const bool sample = (top_k != 0 || top_p != 1.0f) && uniforms != nullptr;
  int token; float conf, prob;
  select_from_logits(lg, srt, V, Vp2, top_k, top_p, sample, sample ? uniforms[b] : 0.f, token, conf, &prob);
  if (threadIdx.x == 0) { if (token_out) token_out[b] = token; if (conf_out) conf_out[b] = conf; if (prob_out) prob_out[b] = prob; }
}

int next_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }

// operand rows of a LayerNorm-on-load / embedding source as IEEE half (+ the f32 residual copy), one warp per image
int launch_prep(mdc_ctx* ctx, const XSrc& xs, __half* xh, int B, int K, cudaStream_t s) {
  const dim3 grid((B + LIN_WARPS - 1) / LIN_WARPS);
  const bool al = (((uintptr_t)xh | (uintptr_t)xs.xn_out | (uintptr_t)xs.resid | (uintptr_t)xs.delta | (uintptr_t)xs.ln_w | (uintptr_t)xs.ln_b |
                    (uintptr_t)xs.emb | (uintptr_t)xs.pos) & 15) == 0;
  if (al && K == 256) prep_x_half_vec_kernel<2><<<grid, LIN_THREADS, 0, s>>>(xs, xh, B);
  else if (al && K == 512) prep_x_half_vec_kernel<4><<<grid, LIN_THREADS, 0, s>>>(xs, xh, B);
  else if (al && K == 1024) prep_x_half_vec_kernel<8><<<grid, LIN_THREADS, 0, s>>>(xs, xh, B);
  else prep_x_half_kernel<<<grid, LIN_THREADS, 0, s>>>(xs, xh, B, K);
  MDC_LAUNCH_CHECK(ctx); return 0;
}

// batches of 16 and more with K a multiple of 256 (eight warps x 32-column blocks) take the weight-streaming linear
inline bool stream_linears(int B, int K) { return B >= 16 && K % 256 == 0; }

template <typename TW>
int launch_linear(mdc_ctx* ctx, const XSrc& xs, const void* W, const float* bias, float* Y, int64_t ldy, int B, int N, int K,
                  bool relu, cudaStream_t s, __half* xh_buf = nullptr, __half* yh = nullptr, int64_t ldyh = 0, int mt2_min_n = STREAM_MT2_MIN_N,
                  const void* next_w = nullptr, size_t next_w_bytes = 0) {
  MDC_CHECK_ARG(K % 8 == 0);
  if constexpr (std::is_same<TW, __half>::value) {
    // weight-streaming form: operand rows available as IEEE half (built here by prep_x_half_kernel, or the producer's half twin)
    if (stream_linears(B, K) && xh_buf && (xs.mode != XMODE_PLAIN || (xs.xh && xs.ldxh % 8 == 0 && ((uintptr_t)xs.xh & 15) == 0))) {
      const __half* X = xs.xh; int64_t ldx = xs.ldxh;
      if (xs.mode != XMODE_PLAIN) {
        MDC_TRY(launch_prep(ctx, xs, xh_buf, B, K, s));
        X = xh_buf; ldx = K;
      }
      const int mt = N >= mt2_min_n ? 2 : 1;
      dim3 grid((N + STREAM_ROWS * mt - 1) / (STREAM_ROWS * mt), (B + MMA_IMGS - 1) / MMA_IMGS);
#define MDC_STREAM(RELU_, MT_)                                                                                                              \
  {                                                                                                                                         \
    MDC_ENSURE_SMEM((dec_linear_stream_kernel<RELU_, MT_>), STREAM_SMEM);                                                                   \
    dec_linear_stream_kernel<RELU_, MT_><<<grid, LIN_THREADS, STREAM_SMEM, s>>>(X, ldx, (const __half*)W, bias, Y, ldy, yh, ldyh, B, N, K,   \
                                                                                (const uint8_t*)next_w, (int)(next_w_bytes / 128), xs.done); \
  }
      if (relu) { if (mt == 2) MDC_STREAM(true, 2) else MDC_STREAM(true, 1) }
      else { if (mt == 2) MDC_STREAM(false, 2) else MDC_STREAM(false, 1) }
#undef MDC_STREAM
      MDC_LAUNCH_CHECK(ctx); return 0;
    }
    MDC_CHECK_ARG(Y != nullptr && yh == nullptr);
    // batches of 16 and more on the tensor cores (weights read once per 64 images); LayerNorm / embedding operands are model-width rows
    const bool plain = xs.mode == XMODE_PLAIN;
    if (xh_buf && B >= 16 && K % 32 == 0 && (plain ? (K <= MMA_KC || K % MMA_KC == 0) && xs.ldx % 4 == 0 && ((uintptr_t)xs.x & 15) == 0 : K <= MMA_KC)) {
      XSrc src = xs;
      if (!plain) {
        MDC_TRY(launch_prep(ctx, xs, xh_buf, B, K, s));
        src = XSrc{}; src.mode = XMODE_HALF; src.xh = xh_buf; src.done = xs.done;
      }
      const size_t sm = (size_t)MMA_IMGS * (size_t)((K < MMA_KC ? K : MMA_KC) + MMA_PAD) * sizeof(__half);
      dim3 grid((N + MMA_ROWS - 1) / MMA_ROWS, (B + MMA_IMGS - 1) / MMA_IMGS);
      if (relu) {
        MDC_ENSURE_SMEM(dec_linear_mma_kernel<true>, sm);
        dec_linear_mma_kernel<true><<<grid, LIN_THREADS, sm, s>>>(src, (const __half*)W, bias, Y, ldy, B, N, K);
      } else {
        MDC_ENSURE_SMEM(dec_linear_mma_kernel<false>, sm);
        dec_linear_mma_kernel<false><<<grid, LIN_THREADS, sm, s>>>(src, (const __half*)W, bias, Y, ldy, B, N, K);
      }
      MDC_LAUNCH_CHECK(ctx); return 0;
    }
  }
  const size_t smem = (size_t)BT * K * sizeof(float);
  dim3 block(LIN_THREADS);
  const int gy = (B + BT - 1) / BT;
#define MDC_LIN(RW_, KCH_)                                                                                            \
  {                                                                                                                   \
    dim3 grid((N + LIN_WARPS * RW_ - 1) / (LIN_WARPS * RW_), gy);                                                     \
    if (relu) {                                                                                                       \
      MDC_ENSURE_SMEM((dec_linear_kernel<TW, RW_, KCH_, true>), smem);                                                \
      dec_linear_kernel<TW, RW_, KCH_, true><<<grid, block, smem, s>>>(xs, (const TW*)W, bias, Y, ldy, B, N);          \
    } else {                                                                                                          \
      MDC_ENSURE_SMEM((dec_linear_kernel<TW, RW_, KCH_, false>), smem);                                               \
      dec_linear_kernel<TW, RW_, KCH_, false><<<grid, block, smem, s>>>(xs, (const TW*)W, bias, Y, ldy, B, N);         \
    }                                                                                                                 \
  }
  const int kch = (K % 256 == 0) ? K / 256 : 0;
  // columns per warp: enough CTAs to cover the SMs, bounded register footprint (RW * KCH <= 8 weight slices)
  if (kch == 1) { if (N >= 1536) MDC_LIN(4, 1) else if (N >= 512) MDC_LIN(2, 1) else MDC_LIN(1, 1) }
  else if (kch == 2) { if (N >= 1536) MDC_LIN(4, 2) else if (N >= 512) MDC_LIN(2, 2) else MDC_LIN(1, 2) }
  else if (kch == 4) { if (N >= 1536) MDC_LIN(2, 4) else MDC_LIN(1, 4) }
  else if (kch == 8) { MDC_LIN(1, 8) }
  else {
    dim3 grid((N + LIN_WARPS - 1) / LIN_WARPS, gy);
    if (relu) {
      MDC_ENSURE_SMEM((dec_linear_generic_kernel<TW, true>), smem);
      dec_linear_generic_kernel<TW, true><<<grid, block, smem, s>>>(xs, (const TW*)W, bias, Y, ldy, B, N, K);
    } else {
      MDC_ENSURE_SMEM((dec_linear_generic_kernel<TW, false>), smem);
      dec_linear_generic_kernel<TW, false><<<grid, block, smem, s>>>(xs, (const TW*)W, bias, Y, ldy, B, N, K);
    }
  }
#undef MDC_LIN
  MDC_LAUNCH_CHECK(ctx); return 0;
}

struct Scratch { float *xa, *xb, *xc, *y1, *y2, *y3, *qkv, *qc, *o, *oc, *f1, *lg; __half *xh, *oh, *f1h; int *fin, *stop_state; };

size_t scratch_floats(const mdc_dims& d, int B) {
  // + the fp16 operand rows of the tensor-core linears (B x dim halves, behind the step logits, 16-byte aligned)
  // + the IEEE-half twins of the attention output and of the FFN hidden (operands of the weight-streaming linears)
  // + the stop-at-EOS words (StopArgs: B finished flags, count, all-finished flag; 16-byte aligned)
  return (size_t)B * ((size_t)d.dim * 9 + (size_t)d.dim * 3 + d.dec_ffn + d.vocab) + 4 + ((size_t)B * d.dim + 1) / 2
         + 8 + ((size_t)B * d.dim + 1) / 2 + ((size_t)B * d.dec_ffn + 1) / 2 + 4 + B + 2;
}

Scratch carve(const mdc_dims& d, int B, void* p) {
  float* f = (float*)p; Scratch s; size_t bd = (size_t)B * d.dim;
  s.xa = f; f += bd; s.xb = f; f += bd; s.xc = f; f += bd; s.y1 = f; f += bd; s.y2 = f; f += bd; s.y3 = f; f += bd;
  s.qc = f; f += bd; s.o = f; f += bd; s.oc = f; f += bd; s.qkv = f; f += 3 * bd; s.f1 = f; f += (size_t)B * d.dec_ffn; s.lg = f; f += (size_t)B * d.vocab;
  s.xh = reinterpret_cast<__half*>((reinterpret_cast<uintptr_t>(f) + 15) & ~(uintptr_t)15);
  s.oh = reinterpret_cast<__half*>((reinterpret_cast<uintptr_t>(s.xh + bd) + 15) & ~(uintptr_t)15);
  s.f1h = reinterpret_cast<__half*>((reinterpret_cast<uintptr_t>(s.oh + bd) + 15) & ~(uintptr_t)15);
  s.fin = reinterpret_cast<int*>((reinterpret_cast<uintptr_t>(s.f1h + (size_t)B * d.dec_ffn) + 15) & ~(uintptr_t)15);
  s.stop_state = s.fin + B;
  return s;
}

// T: element type of the KV caches (`precision`); TW: element type of the decode-loop weights, f32 under fp32 and IEEE half under bf16
template <typename T>
int decode_step_typed(mdc_model* m, const mdc_decode_state* st, int t, cudaStream_t s) {
  using TW = typename std::conditional<std::is_same<T, float>::value, float, __half>::type;
  constexpr bool HALF = std::is_same<TW, __half>::value;
  mdc_ctx* ctx = m->ctx; const mdc_dims& d = m->d;
  const int B = st->B, dim = d.dim, hd = dim / d.dec_heads;
  const void** gw = m->w + MDC_ENC_GLOBAL_SLOTS + d.enc_depth * MDC_ENC_BLOCK_SLOTS;
  const void** lw0 = gw + MDC_DEC_GLOBAL_SLOTS;
  Scratch sc = carve(d, B, st->scratch);
  const float scale = 1.0f / sqrtf((float)hd);
  // wide batches on fp16 decode-loop weights: weight-streaming linears fed with IEEE-half operands by their producers
  const bool stream = HALF && stream_linears(B, dim) && stream_linears(B, d.dec_ffn) && dim % 8 == 0;
  // the batch pipeline asks for 16 images per cluster = "SM-time over latency": there every linear takes two row tiles per CTA (half the
  // CTAs; same bits -- the tile count does not enter any element's arithmetic).  A/B at B = 64: serial token-step +10 %, pipeline +9 %.
  const int mt2 = st->images_per_cluster >= 16 ? 512 : STREAM_MT2_MIN_N;
  const StopArgs stop = st->stop_at_eos ? StopArgs{sc.fin, sc.stop_state, st->eos_token} : StopArgs{nullptr, nullptr, 0};
  const int* done = st->stop_at_eos ? sc.stop_state + 1 : nullptr;
  XSrc prev{};   // how the next consumer obtains the layer input
  prev.done = done;
  if (st->x_override) { prev.mode = XMODE_PLAIN; prev.x = st->x_override + (int64_t)t * dim; prev.ldx = (int64_t)st->x_override_ld * dim; }
  else {
    prev.mode = XMODE_EMBED; prev.tokens = st->tokens; prev.tokens_ld = st->tokens_ld; prev.t = t;
    prev.emb = (const float*)gw[MDC_EMB]; prev.pos = st->pos_override ? st->pos_override : (const float*)gw[MDC_DEC_POS];
  }
  for (int l = 0; l < d.dec_layers; ++l) {
    const void** lw = lw0 + l * MDC_DEC_LAYER_SLOTS;
    // qkv = LNload(prev) . Ws^T + bs; publishes xa
    XSrc x1 = prev; x1.xn_out = sc.xa;
    MDC_TRY(launch_linear<TW>(ctx, x1, lw[MDC_SA_IN_W], (const float*)lw[MDC_SA_IN_B], sc.qkv, 3 * dim, B, 3 * dim, dim, false, s, sc.xh, nullptr, 0, mt2, lw[MDC_SA_OUT_W], (size_t)dim * dim * sizeof(TW)));
    {
      size_t smem = (size_t)d.dec_heads * (hd + t + 1 + st->pages_per_seq) * sizeof(float);
#define MDC_SA(HD_)                                                                                                      \
  {                                                                                                                      \
    MDC_ENSURE_SMEM((dec_self_attn_kernel<T, HD_>), smem);                                                               \
    dec_self_attn_kernel<T, HD_><<<B, d.dec_heads * 32, smem, s>>>(sc.qkv, (T*)st->kv_pool, st->page_table, st->pages_per_seq, \
        d.page_tokens, d.dec_layers, l, st->tokens, st->tokens_ld, d.pad_idx, t, dim, scale, sc.o, stream ? sc.oh : nullptr, done); \
  }
      if (hd == 32) MDC_SA(32) else if (hd == 64) MDC_SA(64) else MDC_SA(128)      // the head widths mdc_model_create accepts
#undef MDC_SA
      MDC_LAUNCH_CHECK(ctx);
    }
    XSrc xo{}; xo.mode = XMODE_PLAIN; xo.x = sc.o; xo.ldx = dim; xo.done = done;
    if (stream) { xo.xh = sc.oh; xo.ldxh = dim; }
    MDC_TRY(launch_linear<TW>(ctx, xo, lw[MDC_SA_OUT_W], (const float*)lw[MDC_SA_OUT_B], sc.y1, dim, B, dim, dim, false, s, sc.xh, nullptr, 0, mt2, lw[MDC_CA_IN_W], (size_t)dim * dim * sizeof(TW)));
    // cross-attention query from LN1(xa + y1); publishes xb
    XSrc x2{}; x2.mode = XMODE_LN; x2.resid = sc.xa; x2.delta = sc.y1; x2.ln_w = (const float*)lw[MDC_LN1_W]; x2.ln_b = (const float*)lw[MDC_LN1_B];
    x2.eps = 1e-5f; x2.xn_out = sc.xb; x2.done = done;
    MDC_TRY(launch_linear<TW>(ctx, x2, lw[MDC_CA_IN_W], (const float*)lw[MDC_CA_IN_B], sc.qc, dim, B, dim, dim, false, s, sc.xh, nullptr, 0, mt2, lw[MDC_CA_OUT_W], (size_t)dim * dim * sizeof(TW)));
    {
      size_t smem = (size_t)d.dec_heads * (hd + d.n_patches) * sizeof(float);
      const T* ckv = (const T*)st->cross_kv + (int64_t)l * B * d.n_patches * 2 * dim;
#define MDC_CA(HD_)                                                                                         \
  {                                                                                                         \
    MDC_ENSURE_SMEM((dec_cross_attn_kernel<T, HD_>), smem);                                                 \
    dec_cross_attn_kernel<T, HD_><<<B, d.dec_heads * 32, smem, s>>>(sc.qc, ckv, d.n_patches, dim, scale, sc.oc, done); \
  }
#define MDC_CAS(HD_)                                                                                        \
  {                                                                                                         \
    const size_t smem_s = (size_t)(HD_ + LIN_WARPS * HD_ + 2 * LIN_WARPS + d.n_patches) * sizeof(float);   \
    MDC_ENSURE_SMEM((dec_cross_attn_split_kernel<T, HD_>), smem_s);                                         \
    dec_cross_attn_split_kernel<T, HD_><<<dim3(d.dec_heads, B), LIN_THREADS, smem_s, s>>>(sc.qc, ckv, d.n_patches, dim, scale, sc.oh, done); \
  }
      if (stream) { if constexpr (HALF) { if (hd == 32) MDC_CAS(32) else if (hd == 64) MDC_CAS(64) else MDC_CAS(128) } }
      else if (hd == 32) MDC_CA(32) else if (hd == 64) MDC_CA(64) else MDC_CA(128)
#undef MDC_CA
#undef MDC_CAS
      MDC_LAUNCH_CHECK(ctx);
    }
    XSrc xco{}; xco.mode = XMODE_PLAIN; xco.x = sc.oc; xco.ldx = dim; xco.done = done;
    if (stream) { xco.xh = sc.oh; xco.ldxh = dim; }
    MDC_TRY(launch_linear<TW>(ctx, xco, lw[MDC_CA_OUT_W], (const float*)lw[MDC_CA_OUT_B], sc.y2, dim, B, dim, dim, false, s, sc.xh, nullptr, 0, mt2, lw[MDC_FF1_W], (size_t)d.dec_ffn * dim * sizeof(TW)));
    // FFN
    XSrc x3{}; x3.mode = XMODE_LN; x3.resid = sc.xb; x3.delta = sc.y2; x3.ln_w = (const float*)lw[MDC_LN2_W]; x3.ln_b = (const float*)lw[MDC_LN2_B];
    x3.eps = 1e-5f; x3.xn_out = sc.xc; x3.done = done;
    if (stream) MDC_TRY(launch_linear<TW>(ctx, x3, lw[MDC_FF1_W], (const float*)lw[MDC_FF1_B], nullptr, 0, B, d.dec_ffn, dim, true, s, sc.xh, sc.f1h, d.dec_ffn, mt2, lw[MDC_FF2_W], (size_t)d.dec_ffn * dim * sizeof(TW)));
    else MDC_TRY(launch_linear<TW>(ctx, x3, lw[MDC_FF1_W], (const float*)lw[MDC_FF1_B], sc.f1, d.dec_ffn, B, d.dec_ffn, dim, true, s, sc.xh, nullptr, 0, mt2));
    XSrc xf{}; xf.mode = XMODE_PLAIN; xf.x = sc.f1; xf.ldx = d.dec_ffn; xf.done = done;
    // what the linear after FFN2 streams: the next layer's in-projection, or the vocabulary head
    const void* next_in_w = l + 1 < d.dec_layers ? (lw + MDC_DEC_LAYER_SLOTS)[MDC_SA_IN_W] : gw[MDC_OUT_W];
    const size_t next_in_bytes = l + 1 < d.dec_layers ? 3 * (size_t)dim * dim * sizeof(TW) : (size_t)d.vocab * dim * sizeof(TW);
    if (stream) { xf.xh = sc.f1h; xf.ldxh = d.dec_ffn; }
    MDC_TRY(launch_linear<TW>(ctx, xf, lw[MDC_FF2_W], (const float*)lw[MDC_FF2_B], sc.y3, dim, B, dim, d.dec_ffn, false, s, sc.xh, nullptr, 0, mt2, next_in_w, next_in_bytes));
    prev = XSrc{}; prev.mode = XMODE_LN; prev.resid = sc.xc; prev.delta = sc.y3; prev.ln_w = (const float*)lw[MDC_LN3_W];
    prev.ln_b = (const float*)lw[MDC_LN3_B]; prev.eps = 1e-5f; prev.done = done;
  }
  {
    const int V = d.vocab, Vp2 = next_pow2(V);
    MDC_TRY(launch_linear<TW>(ctx, prev, gw[MDC_OUT_W], (const float*)gw[MDC_OUT_B], sc.lg, V, B, V, dim, false, s, sc.xh, nullptr, 0, mt2, lw0[MDC_SA_IN_W], 3 * (size_t)dim * dim * sizeof(TW)));
    size_t smem = (size_t)(V + Vp2) * sizeof(float);
    MDC_ENSURE_SMEM(dec_select_kernel, smem);
    dec_select_kernel<<<B, SEL_THREADS, smem, s>>>(sc.lg, V, Vp2, t, st->logits, (int64_t)st->logits_ld * V, t + st->logits_row_offset,
                                                  st->tokens, st->tokens_ld, st->forced, st->confs, st->confs_ld, st->uniforms,
                                                  st->uniforms_ld, st->top_k, st->top_p, stop);
    MDC_LAUNCH_CHECK(ctx);
  }
  return 0;
}

}  // namespace

extern "C" size_t mdc_decode_workspace_bytes(const mdc_model* m, int B) {
  if (!m || B <= 0) return 0;
  return align_up(scratch_floats(m->d, B) * sizeof(float), 256);
}

extern "C" size_t mdc_kv_page_bytes(const mdc_model* m) {
  if (!m) return 0;
  return (size_t)m->d.dec_layers * 2 * m->d.page_tokens * m->d.dim * esize(m->d.precision);
}

extern "C" int mdc_decode_steps(mdc_model* m, const mdc_decode_state* st, int t_begin, int t_end, void* stream) {
  MDC_CHECK_ARG(m && st && st->B > 0 && st->tokens && st->kv_pool && st->page_table && st->cross_kv && st->scratch);
  MDC_CHECK_DEVICE(m->ctx);
  MDC_CHECK_ARG(t_begin >= 0 && t_end >= t_begin);
  MDC_CHECK_ARG(st->x_override || st->pos_override || t_end <= m->d.max_pos);   // Q6: the pos table has max_len-1 rows
  MDC_CHECK_ARG(t_end <= st->pages_per_seq * m->d.page_tokens);
  MDC_CHECK_ARG(st->forced || t_end < st->tokens_ld);
  MDC_CHECK_ARG(st->scratch_bytes >= mdc_decode_workspace_bytes(m, st->B));
  if (st->logits) MDC_CHECK_ARG(t_end + st->logits_row_offset <= st->logits_ld);
  if (st->confs) MDC_CHECK_ARG((t_end + 3) / 4 <= st->confs_ld);
  if ((st->top_k != 0 || st->top_p != 1.0f) && !st->forced) MDC_CHECK_ARG(st->uniforms && t_end <= st->uniforms_ld);
  if (st->stop_at_eos) MDC_CHECK_ARG(!st->forced && !st->logits && st->eos_token >= 0 && st->eos_token < m->d.vocab);
  cudaStream_t s = (cudaStream_t)stream;
  if (t_end > t_begin && decode_cluster_supported(m, st, t_end)) {
    Scratch sc = carve(m->d, st->B, st->scratch);      // the cluster kernel only needs the step-logits area
    return decode_cluster_launch(m, st, t_begin, t_end, sc.lg, s);
  }
  if (st->stop_at_eos && t_end > t_begin) {
    Scratch sc = carve(m->d, st->B, st->scratch);
    dec_stop_init_kernel<<<1, SEL_THREADS, 0, s>>>(st->tokens, st->tokens_ld, st->confs, st->confs_ld, st->B, t_begin, t_end, m->d.pad_idx,
                                                   StopArgs{sc.fin, sc.stop_state, st->eos_token});
    MDC_LAUNCH_CHECK(m->ctx);
  }
  for (int t = t_begin; t < t_end; ++t) {
    if (m->d.precision == MDC_F32) MDC_TRY(decode_step_typed<float>(m, st, t, s));
    else MDC_TRY(decode_step_typed<bf16>(m, st, t, s));
  }
  return 0;
}

extern "C" int mdc_select(mdc_ctx* ctx, const float* logits, int64_t ld, int B, int V, int top_k, float top_p, const float* uniforms,
                          int32_t* token_out, float* conf_out, float* prob_out, void* stream) {
  MDC_CHECK_ARG(ctx && logits && B > 0 && V > 0 && V <= 4096 && (token_out || conf_out || prob_out));
  MDC_CHECK_DEVICE(ctx);
  int Vp2 = next_pow2(V);
  size_t smem = (size_t)(V + Vp2) * sizeof(float);
  select_kernel<<<B, SEL_THREADS, smem, (cudaStream_t)stream>>>(logits, ld, V, Vp2, top_k, top_p, uniforms, token_out, conf_out, prob_out);
  MDC_LAUNCH_CHECK(ctx); return 0;
}
