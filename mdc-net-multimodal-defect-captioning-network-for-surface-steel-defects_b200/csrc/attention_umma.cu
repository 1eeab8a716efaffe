// attention_umma.cu -- strip attention of the ViT blocks on the 5th-generation tensor cores (tcgen05 / TMEM / TMA), bf16, head width 64,
// strips of up to 256 tokens (the 197-token strips of 224x224 inputs; longer strips stay on attention_tc.cu's chunked mma.sync kernel).
//
// One persistent CTA per SM walks (strip, head) items.  Per item:
//   TMA        Q (256 rows), K and V (NK = roundup16(S) rows) head slices of the packed qkv matrix -> shared memory, 128-byte rows,
//              SWIZZLE_128B, double buffered across items
//   tcgen05    S = Q K^T per 128-query tile: 4 x UMMA 128 x NK x 16 (K-major operands), fp32 accumulators in TMEM
//   softmax    16 warps, four threads per query row (each holds a quarter of the row's NK scores in registers: ONE tcgen05.ld pass), row
//              max exchanged through shared memory, exp2 in the log2 domain (MUFU-bound: 4 lanes per clock and sub-partition), P
//              written back to TMEM IN PLACE as packed bf16
//   tcgen05    O = P V: A operand = P straight from TMEM, B operand = V as it lies in shared memory ([key][dim] rows = MN-major,
//              instruction-descriptor transpose bit), 13 x UMMA 128 x 64 x 16
//   epilogue   O from TMEM, scaled by 1 / row sum, bf16, one 64-byte store per thread
// The two query tiles of a strip overlap: while the softmax warps work on tile 1 the tensor core runs P V of tile 0.
// TMEM columns of tile t (256-column region): S in [0, NK), P overwrites [0, NK/2) once S is in registers, O goes to [128, 192).
#include "common.cuh"
#include <cuda.h>
#include <stdlib.h>

namespace {

constexpr int HD = 64;
constexpr int QROWS = 256;                 // query rows staged per item (two 128-row MMA tiles)
constexpr int N_SOFTMAX_WARPS = 16;
constexpr int THREADS = 64 + N_SOFTMAX_WARPS * 32;

struct SmemLayout {          // per item buffer: Q | K | V, each 1024-aligned
  int q_bytes, kv_bytes, buf_bytes;
};

__global__ void __launch_bounds__(THREADS, 1)
attn_umma_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_kv, bf16* __restrict__ out, int64_t ldo,
                 int n_items, int S, int H, int NK, float scale_log2e, long long* dbg) {
#ifdef MDC_DEVTOOLS
#define STAMP(i) do { if (dbg && blockIdx.x == 0 && n == 0) dbg[i] = clock64(); } while (0)
#else
#define STAMP(i) do { } while (0)
#endif
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const int q_bytes = QROWS * 128, kv_bytes = NK * 128, buf_bytes = q_bytes + 2 * kv_bytes;      // NK % 16 == 0: kv_bytes % 2048 == 0
  uint64_t* bars = (uint64_t*)(smem + 2 * buf_bytes);
  // barriers: full[2], sfree[2], s_ready[2], p_ready[2], o_ready[2], t_free[2]
  uint64_t* full = bars; uint64_t* sfree = bars + 2; uint64_t* s_ready = bars + 4; uint64_t* p_ready = bars + 6; uint64_t* o_ready = bars + 8;
  uint64_t* t_free = bars + 10;
  uint32_t* tmem_ptr_smem = (uint32_t*)(bars + 12);
  float* xch = (float*)(bars + 16);                 // [4 parts][128 rows] row maxima, then per tile [4][128] row sums
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles = S > 128 ? 2 : 1;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&full[i]), 1); mbar_init(smem_u32(&sfree[i]), 1); mbar_init(smem_u32(&s_ready[i]), 1);
      mbar_init(smem_u32(&p_ready[i]), N_SOFTMAX_WARPS * 32); mbar_init(smem_u32(&o_ready[i]), 1); mbar_init(smem_u32(&t_free[i]), N_SOFTMAX_WARPS * 32);
    }
    fence_mbarrier_init();
    prefetch_tmap(&map_q);
    prefetch_tmap(&map_kv);
  }
  if (warp == 0) {
    tmem_alloc<1>(smem_u32(tmem_ptr_smem), 512);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  const int D = H * HD;

  if (warp == 1) {
    // ===== TMA producer =====
    if (lane == 0) {
      int n = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++n) {
        const int buf = n & 1, strip = item / H, head = item % H;
        mbar_wait(smem_u32(&sfree[buf]), ((n >> 1) & 1) ^ 1);
        const uint32_t fb = smem_u32(&full[buf]);
        const uint32_t base = smem_u32(smem + buf * buf_bytes);
        STAMP(0);
        mbar_expect_tx(fb, (uint32_t)(3 * kv_bytes));       // Q, K, V: NK rows each (query rows beyond NK of the second tile stay stale: never stored)
        tma_load_2d(&map_kv, fb, base, head * HD, strip * S);
        tma_load_2d(&map_kv, fb, base + q_bytes, D + head * HD, strip * S);
        tma_load_2d(&map_kv, fb, base + q_bytes + kv_bytes, 2 * D + head * HD, strip * S);
      }
    }
  } else if (warp == 0) {
    // ===== MMA issuer (one thread) =====
    if (lane == 0) {
      const uint32_t idesc_qk = make_idesc(128, NK), idesc_pv = make_idesc(128, HD, false, true);
      int n = 0;
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++n) {
        const int buf = n & 1;
        const uint32_t base = smem_u32(smem + buf * buf_bytes);
        mbar_wait(smem_u32(&full[buf]), (n >> 1) & 1);
        STAMP(1);
        tc_fence_after();
        const uint64_t kdesc = make_sw128_desc(base + q_bytes);
        for (int t = 0; t < tiles; ++t) {
          mbar_wait(smem_u32(&t_free[t]), (n & 1) ^ 1);           // the previous item's epilogue has drained this tile's TMEM region
          tc_fence_after();
          const uint64_t qdesc = make_sw128_desc(base + t * 128 * 128);
#pragma unroll
          for (int k = 0; k < HD / 16; ++k) umma_ss(tmem_base + t * 256, qdesc + 2 * k, kdesc + 2 * k, idesc_qk, k != 0);
          umma_commit(smem_u32(&s_ready[t]));
          STAMP(2 + t);
        }
        const uint64_t vdesc = make_sw128_desc(base + q_bytes + kv_bytes);
        for (int t = 0; t < tiles; ++t) {
          mbar_wait(smem_u32(&p_ready[t]), n & 1);
          STAMP(4 + t);
          tc_fence_after();
          for (int k = 0; k < NK / 16; ++k)                       // P: 8 packed columns per 16 keys; V: 16 key rows = 2048 bytes
            umma_ts(tmem_base + t * 256 + 128, tmem_base + t * 256 + 8 * k, vdesc + (uint64_t)(128 * k), idesc_pv, k != 0);
          umma_commit(smem_u32(&o_ready[t]));
          STAMP(6 + t);
        }
        umma_commit(smem_u32(&sfree[buf]));                       // every MMA that reads this buffer has completed when this arrives
      }
    }
  } else {
    // ===== softmax + epilogue warps: thread = (query row of the tile, column quarter) =====
    // 16 warps: warp w may touch TMEM lanes [32 (w % 4), +32); the four warps of a lane quarter split the NK score columns four ways
    // (NK / 4 <= 64 scores per thread, held in registers between the max and the exp pass: one tcgen05.ld pass over S).
    const int sw = warp - 2, part = sw >> 2, row = 32 * (warp & 3) + lane;
    const int qc = NK / 4;                          // score columns per thread (multiple of 4, <= 64)
    const int nch = qc / 4;
    const uint32_t lane_addr = (uint32_t)(32 * (warp & 3)) << 16;
    int n = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++n) {
      const int strip = item / H, head = item % H;
      float rsum[2] = {0.f, 0.f};
      for (int t = 0; t < tiles; ++t) {
        mbar_wait(smem_u32(&s_ready[t]), n & 1);
        if (threadIdx.x == 64) STAMP(10 + 8 * t);
        tc_fence_after();
        const uint32_t trow = tmem_base + lane_addr + t * 256;
        // rows beyond the strip's end (the second tile of a 197-token strip has 59): a warp without a valid row skips the arithmetic --
        // its P stays stale and feeds only its own output rows, which are never stored
        const bool live = __any_sync(0xffffffffu, t * 128 + row < S);
        float s[64];
        if (live) {
          // the widest tcgen05.ld shapes that cover the thread's qc = 4 nch columns (52 = 32 + 16 + 4 for 197-token strips): thirteen
          // 4-column loads per thread took 1600 cycles per tile -- bound by the number of TMEM load instructions, not by their bytes
          uint32_t* sr = reinterpret_cast<uint32_t*>(s);
          const uint32_t tcol = trow + part * qc;
          if (nch >= 8) {
            tmem_ld32(tcol, sr);
            if (nch == 16) tmem_ld32(tcol + 32, sr + 32);
            else if (nch >= 12) {
              tmem_ld16(tcol + 32, sr + 32);
#pragma unroll
              for (int c = 12; c < 15; ++c) if (c < nch) tmem_ld4(tcol + 4 * c, sr + 4 * c);
            } else {
#pragma unroll
              for (int c = 8; c < 11; ++c) if (c < nch) tmem_ld4(tcol + 4 * c, sr + 4 * c);
            }
          } else if (nch >= 4) {
            tmem_ld16(tcol, sr);
#pragma unroll
            for (int c = 4; c < 7; ++c) if (c < nch) tmem_ld4(tcol + 4 * c, sr + 4 * c);
          } else {
#pragma unroll
            for (int c = 0; c < 3; ++c) if (c < nch) tmem_ld4(tcol + 4 * c, sr + 4 * c);
          }
          tmem_ld_wait();
        }
        if (threadIdx.x == 64) STAMP(11 + 8 * t);
        // raw scores; scale > 0, so the maximum of the raw scores is the maximum of the scaled ones.  Only the chunk that straddles the
        // strip's end pays for masking.
        const int nvalid = min(max(S - part * qc, 0), qc);       // valid score columns of this thread's part
        float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
        if (live) {
#pragma unroll
          for (int c = 0; c < 16; ++c)
            if (c < nch) {
              if (4 * c + 4 <= nvalid) {
#pragma unroll
                for (int j = 0; j < 4; ++j) m4[j] = fmaxf(m4[j], s[4 * c + j]);
              } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  if (4 * c + j >= nvalid) s[4 * c + j] = -INFINITY;
                  m4[j] = fmaxf(m4[j], s[4 * c + j]);
                }
              }
            }
        }
        float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
        xch[part * 128 + row] = mx;
        bar_sync<128>(1 + (warp & 3));       // the four warps of this lane quarter: every part of these rows has its scores in registers
        if (threadIdx.x == 64) STAMP(12 + 8 * t);
        mx = fmaxf(fmaxf(xch[row], xch[128 + row]), fmaxf(xch[256 + row], xch[384 + row]));      // finite: column 0 is a valid key
        const float nms = -mx * scale_log2e;
        float s4[4] = {0.f, 0.f, 0.f, 0.f};
        if (live) {
#pragma unroll
          for (int c = 0; c < 16; ++c)
            if (c < nch) {
              float p[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) { p[j] = ex2_approx(fmaf(s[4 * c + j], scale_log2e, nms)); s4[j] += p[j]; }
              tmem_st2(trow + (part * qc) / 2 + 2 * c, pack_bf16x2(p[0], p[1]), pack_bf16x2(p[2], p[3]));
            }
        }
        const float sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
        rsum[t] = sum;
        xch[512 + t * 512 + part * 128 + row] = sum;
        if (threadIdx.x == 64) STAMP(13 + 8 * t);
        tmem_st_wait();
        if (threadIdx.x == 64) STAMP(14 + 8 * t);
        tc_fence_before();
        mbar_arrive(smem_u32(&p_ready[t]));
        bar_sync<128>(1 + (warp & 3));       // the maxima in xch are reused by the next tile
      }
      for (int t = 0; t < tiles; ++t) {
        mbar_wait(smem_u32(&o_ready[t]), n & 1);
        if (threadIdx.x == 64) STAMP(26 + 2 * t);
        tc_fence_after();
        const uint32_t trow = tmem_base + lane_addr + t * 256 + 128;
        uint32_t o[16];
        tmem_ld16(trow + part * 16, o);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(smem_u32(&t_free[t]));                  // this thread's part of the tile's TMEM region is in registers
        const float* sx = xch + 512 + t * 512 + row;
        const float inv = 1.0f / ((sx[0] + sx[128]) + (sx[256] + sx[384]));
        const int q = t * 128 + row;
        if (q < S) {
          bf16* dst = out + ((int64_t)strip * S + q) * ldo + head * HD + part * 16;
#pragma unroll
          for (int j = 0; j < 16; j += 8) {
            uint4 v;
            v.x = pack_bf16x2(__uint_as_float(o[j]) * inv, __uint_as_float(o[j + 1]) * inv);
            v.y = pack_bf16x2(__uint_as_float(o[j + 2]) * inv, __uint_as_float(o[j + 3]) * inv);
            v.z = pack_bf16x2(__uint_as_float(o[j + 4]) * inv, __uint_as_float(o[j + 5]) * inv);
            v.w = pack_bf16x2(__uint_as_float(o[j + 6]) * inv, __uint_as_float(o[j + 7]) * inv);
            *reinterpret_cast<uint4*>(dst + j) = v;
          }
        }
      }
      if (threadIdx.x == 64) STAMP(30);
      bar_sync<128>(1 + (warp & 3));         // the row sums in xch are reused by the next item
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, 512);
  }
}

}  // namespace

int attn_umma_supported(int strip_len, int head_dim, int64_t ld, int64_t ldo) {
  return head_dim == HD && strip_len >= 16 && strip_len <= 256 && ld % 8 == 0 && ldo % 8 == 0;
}

int attn_umma_launch(mdc_ctx* ctx, const void* qkv, int64_t ld, void* out, int64_t ldo, int n_strips, int strip_len, int heads, float scale,
                     cudaStream_t s) {
  MDC_CHECK_ARG(((uintptr_t)qkv & 15) == 0 && ((uintptr_t)out & 15) == 0);
  const int S = strip_len, NK = ((S + 15) / 16) * 16;
  const int64_t rows = (int64_t)n_strips * S;
  CUtensorMap mq, mkv;
  // one tensor map over the packed qkv matrix (box = NK rows x 64 columns); the column coordinate selects q / k / v and the head
  MDC_TRY(mdc_make_tmap_2d(ctx, qkv, rows, 3 * heads * HD, ld, HD, NK, 3, &mkv));
  mq = mkv;
  const int buf_bytes = QROWS * 128 + 2 * NK * 128;
  const size_t smem = 2 * (size_t)buf_bytes + 1024 + 128 + 3 * 512 * 4;
  MDC_ENSURE_SMEM(attn_umma_kernel, smem);
  const int n_items = n_strips * heads;
  const int grid = n_items < ctx->sm_count ? n_items : ctx->sm_count;
  long long* dbg = nullptr;
#ifdef MDC_DEVTOOLS
  if (const char* e = getenv("MDC_ATTN_TRACE_PTR")) dbg = (long long*)strtoull(e, nullptr, 0);
#endif
  attn_umma_kernel<<<grid, THREADS, smem, s>>>(mq, mkv, (bf16*)out, ldo, n_items, S, heads, NK, scale * LOG2E, dbg);
  MDC_LAUNCH_CHECK(ctx);
  return 0;
}
