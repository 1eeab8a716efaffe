// attention_tc.cu -- strip attention on the tensor cores for bf16, head_dim 64 (the ViT blocks: 197-token strips;
// also any strip of <= 512 tokens, e.g. 14-token axial strips).
//
// One CTA = one (strip, head): the strip's K and V panels are staged ONCE in shared memory (XOR-swizzled 128-byte
// rows, conflict-free for ldmatrix), one warp per 16 queries.  Per 16-key block a warp issues
//   S = Q.K^T   (mma.sync m16n8k16, Q fragments live in registers for the whole kernel)
//   online softmax in the exp2 domain, row max / sum reduced with quad shuffles
//   O += P.V    (P re-used straight from the S accumulator registers as the A operand; V via ldmatrix.trans)
// so scores and probabilities never leave registers.
#include "common.cuh"

namespace {

constexpr int HD = 64;

// One CTA = one (strip, head, chunk of up to 208 queries): 13 warps x 16 queries, compiled for TWO CTAs per SM (<= 72 registers), so
// one CTA's K/V fetch overlaps the other's MMAs.  Keys are consumed in chunks of up to 208 staged in shared memory (a 197-token
// ViT strip is one chunk and one query chunk -- the common case; a 1025-token strip of a 512x512 input is 5 x 5), the online
// softmax state lives in registers across the chunks.
constexpr int QCHUNK = 208;
template <bool MULTI>      // MULTI = false: the strip is one key chunk and one query chunk (compile-time single trip)
__global__ void __launch_bounds__(416, 2)
attn_tc_kernel(const bf16* __restrict__ qkv, int64_t ld, bf16* __restrict__ out, int64_t ldo, int S, int H, float scale_log2e, int KC) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* Ks = smem; uint8_t* Vs = smem + (size_t)KC * 128;
  const int strip = blockIdx.y, head = blockIdx.x;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bf16* base = qkv + (int64_t)strip * S * ld + head * HD;
  const int D = H * HD;
  const uint32_t ks_u32 = smem_u32(Ks), vs_u32 = smem_u32(Vs);
  // Q fragments straight from global memory (A operand layout of m16n8k16)
  const int q0 = blockIdx.z * QCHUNK + warp * 16, r0 = q0 + (lane >> 2), r1 = r0 + 8;
  const bool active = q0 < S;           // warps past the strip's end only help staging
  uint32_t qa[4][4];
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    const int k = ks * 16 + 2 * (lane & 3);
    qa[ks][0] = r0 < S ? *reinterpret_cast<const uint32_t*>(base + (int64_t)r0 * ld + k) : 0u;
    qa[ks][1] = r1 < S ? *reinterpret_cast<const uint32_t*>(base + (int64_t)r1 * ld + k) : 0u;
    qa[ks][2] = r0 < S ? *reinterpret_cast<const uint32_t*>(base + (int64_t)r0 * ld + k + 8) : 0u;
    qa[ks][3] = r1 < S ? *reinterpret_cast<const uint32_t*>(base + (int64_t)r1 * ld + k + 8) : 0u;
  }
  const uint32_t ks_base = ks_u32, vs_base = vs_u32;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  float o[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) { o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f; }
  for (int kc0 = 0; kc0 < (MULTI ? S : 1); kc0 += KC) {
  // K / V chunk: 16-byte asynchronous copies straight into the swizzled rows (no register staging: every copy of the CTA is in
  // flight at once); rows past the strip's end are zero (they meet p = 0, so they must be finite)
  if (kc0 > 0) __syncthreads();                // every warp is done with the previous chunk
  for (int i = tid; i < KC * 8; i += blockDim.x) {
    const int r = i >> 3, c = i & 7, gr = kc0 + r;
    if (gr < S) {
      cp_async16(ks_u32 + swz<HD>(r, c), base + (int64_t)gr * ld + D + c * 8);
      cp_async16(vs_u32 + swz<HD>(r, c), base + (int64_t)gr * ld + 2 * D + c * 8);
    } else {
      *reinterpret_cast<uint4*>(Ks + swz<HD>(r, c)) = make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4*>(Vs + swz<HD>(r, c)) = make_uint4(0, 0, 0, 0);
    }
  }
  cp_async_wait_all();
  __syncthreads();
  const int nblk = active ? (min(KC, S - kc0) + 15) / 16 : 0;
  for (int kb = 0; kb < nblk; ++kb) {
    const int lk0 = kb * 16, key0 = kc0 + lk0;
    // ---- S = Q K^T for 16 keys: two n-tiles (keys key0..+7, key0+8..+15) ------------------------------------
    float s[2][4] = {{0, 0, 0, 0}, {0, 0, 0, 0}};
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
#pragma unroll
      for (int kp = 0; kp < 2; ++kp) {        // two k-steps (32 dims) per ldmatrix.x4
        // matrices: (dims 32kp..+7), (+8..15), (+16..23), (+24..31) of keys key0+8nt+0..7
        const int krow = lk0 + nt * 8 + (lane & 7), chunk = kp * 4 + (lane >> 3);
        uint32_t kf[4];
        ldsm_x4(kf, ks_base + swz<HD>(krow, chunk));
        mma_m16n8k16<bf16>(s[nt], qa[2 * kp], kf[0], kf[1]);
        mma_m16n8k16<bf16>(s[nt], qa[2 * kp + 1], kf[2], kf[3]);
      }
    }
    // ---- mask + online softmax (exp2 domain) ------------------------------------------------------------------
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      const int kc = key0 + nt * 8 + 2 * (lane & 3);
      if (kc >= S) { s[nt][0] = -INFINITY; s[nt][2] = -INFINITY; }
      if (kc + 1 >= S) { s[nt][1] = -INFINITY; s[nt][3] = -INFINITY; }
    }
    float mx0 = fmaxf(fmaxf(s[0][0], s[0][1]), fmaxf(s[1][0], s[1][1]));
    float mx1 = fmaxf(fmaxf(s[0][2], s[0][3]), fmaxf(s[1][2], s[1][3]));
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);          // finite: key 0 of the first block is always valid
    const float c0 = ex2_approx((m0 - mn0) * scale_log2e), c1 = ex2_approx((m1 - mn1) * scale_log2e);
    m0 = mn0; m1 = mn1;
    const float ms0 = mn0 * scale_log2e, ms1 = mn1 * scale_log2e;
    float p[2][4];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      p[nt][0] = ex2_approx(fmaf(s[nt][0], scale_log2e, -ms0)); p[nt][1] = ex2_approx(fmaf(s[nt][1], scale_log2e, -ms0));
      p[nt][2] = ex2_approx(fmaf(s[nt][2], scale_log2e, -ms1)); p[nt][3] = ex2_approx(fmaf(s[nt][3], scale_log2e, -ms1));
    }
    l0 = l0 * c0 + (p[0][0] + p[0][1]) + (p[1][0] + p[1][1]);
    l1 = l1 * c1 + (p[0][2] + p[0][3]) + (p[1][2] + p[1][3]);
    if (__any_sync(0xffffffffu, c0 != 1.0f || c1 != 1.0f)) {       // a running maximum moved: rescale (rare after the first key blocks)
#pragma unroll
      for (int i = 0; i < 8; ++i) { o[i][0] *= c0; o[i][1] *= c0; o[i][2] *= c1; o[i][3] *= c1; }
    }
    // ---- O += P V : P is the A operand (rows = queries, k = these 16 keys) -----------------------------------------
    uint32_t pa[4];
    pa[0] = pack_bf16x2(p[0][0], p[0][1]); pa[1] = pack_bf16x2(p[0][2], p[0][3]);
    pa[2] = pack_bf16x2(p[1][0], p[1][1]); pa[3] = pack_bf16x2(p[1][2], p[1][3]);
#pragma unroll
    for (int dp = 0; dp < 4; ++dp) {           // two 8-wide dim tiles per ldmatrix.x4.trans
      // matrices: (keys key0..+7, dims 16dp..+7), (keys +8..15, same dims), (keys key0..+7, dims 16dp+8..), (keys +8..15, dims 16dp+8..)
      const int vrow = lk0 + (lane & 7) + ((lane >> 3) & 1) * 8, chunk = dp * 2 + (lane >> 4);
      uint32_t vf[4];
      ldsm_x4_trans(vf, vs_base + swz<HD>(vrow, chunk));
      mma_m16n8k16<bf16>(o[2 * dp], pa, vf[0], vf[1]);
      mma_m16n8k16<bf16>(o[2 * dp + 1], pa, vf[2], vf[3]);
    }
  }
  }
  if (!active) return;
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.0f / l0, i1 = 1.0f / l1;
  bf16* ob = out + (int64_t)strip * S * ldo + head * HD + 2 * (lane & 3);
#pragma unroll
  for (int dt = 0; dt < 8; ++dt) {
    if (r0 < S) *reinterpret_cast<uint32_t*>(ob + (int64_t)r0 * ldo + dt * 8) = pack_bf16x2(o[dt][0] * i0, o[dt][1] * i0);
    if (r1 < S) *reinterpret_cast<uint32_t*>(ob + (int64_t)r1 * ldo + dt * 8) = pack_bf16x2(o[dt][2] * i1, o[dt][3] * i1);
  }
}

}  // namespace

int attn_tc_supported(int strip_len, int head_dim) { return head_dim == HD && strip_len >= 1; }

int attn_tc_launch(mdc_ctx* ctx, const void* qkv, int64_t ld, void* out, int64_t ldo, int n_strips, int strip_len, int heads,
                   int head_dim, float scale, cudaStream_t s) {
  MDC_CHECK_ARG(head_dim == HD && ld % 8 == 0 && ldo % 2 == 0);
  MDC_CHECK_ARG(((uintptr_t)qkv & 15) == 0 && ((uintptr_t)out & 3) == 0);
  const int rows = ((strip_len + 15) / 16) * 16;
  const int KC = rows < QCHUNK ? rows : QCHUNK;                 // keys staged per chunk
  const int q_chunks = (strip_len + QCHUNK - 1) / QCHUNK;
  const size_t smem = (size_t)KC * 128 * 2;
  dim3 grid(heads, n_strips, q_chunks), block(32 * (KC / 16));
  if (q_chunks == 1) {
    MDC_ENSURE_SMEM(attn_tc_kernel<false>, smem);
    attn_tc_kernel<false><<<grid, block, smem, s>>>((const bf16*)qkv, ld, (bf16*)out, ldo, strip_len, heads, scale * LOG2E, KC);
  } else {
    MDC_ENSURE_SMEM(attn_tc_kernel<true>, smem);
    attn_tc_kernel<true><<<grid, block, smem, s>>>((const bf16*)qkv, ld, (bf16*)out, ldo, strip_len, heads, scale * LOG2E, KC);
  }
  MDC_LAUNCH_CHECK(ctx);
  return 0;
}
