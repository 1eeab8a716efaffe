// gemm_tcgen05.cu -- bf16 GEMM D = epi(A[M,K] . W[N,K]^T) on the 5th-gen tensor cores (north_star (a)).
//
//   * persistent: one CTA per SM walks output tiles (n fastest so neighbouring CTAs share the A panel in L2)
//   * warp-specialised: warp 0 = TMA producer (cp.async.bulk.tensor, SWIZZLE_128B, OOB rows/cols zero-filled),
//     warp 1 = MMA issuer (one elected lane issues tcgen05.mma.cta_group::1.kind::f16, 128 x BN x 16),
//     warps 2..9 = epilogue (tcgen05.ld 32x32b from TMEM -> bias / GELU / ReLU / LayerScale+residual / patch+pos);
//     two warps per TMEM lane quadrant split the tile's columns, bias/gamma are staged in shared memory per tile
//     and residual reads are issued before the TMEM read so no global-load latency sits on the critical path
//   * three mbarrier pipelines: smem full/empty (kStages deep), TMEM full/empty (2 accumulator stages, so the
//     epilogue of tile i overlaps the main loop of tile i+1)
//   * accumulators live in TMEM (2 x BN fp32 columns), never in registers.
// Both operands are K-major (A row-major [M,K]; W in nn.Linear layout [N,K]), one 128-byte swizzle atom per
// BLOCK_K = 64 bf16.
#include "common.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>
#include <mutex>
#include <unordered_map>
#include <string.h>
#include <stdlib.h>

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;           // 64 bf16 = 128 B = one SWIZZLE_128B atom
constexpr int UMMA_K = 16;
// warp0 TMA, warp1 MMA, then EW epilogue warps: 8 (two per TMEM lane quadrant) or 16 (four per quadrant, for the 256-wide tiles
// whose epilogue -- GELU over 128 x 256 values -- otherwise outlasts the tile's main loop at two warps per scheduler)

// CTAS = 2: a cluster of two CTAs computes a 256 x BN tile with tcgen05.mma.cta_group::2 -- each CTA stages its own 128 rows of A and
// only HALF of the B tile (BN/2 rows of W); the pair's MMAs read both halves.  A third less shared-memory traffic per flop on both
// sides (TMA writes and tensor-core operand reads): with one CTA per tile the 128 x 256 x 16 MMAs read 12 KB of operands each while the
// TMA unit writes as much -- together with the epilogue's staging that is all of the 128 B/clk shared-memory pipe (ncu: tc + lsu
// wavefronts + the TMA fills = ~100 % of the active cycles; the dev switches MDC_GEMM_DBG show any two of {loads, MMAs, epilogue}
// running at the MMA-only rate and the three together 30 % slower).
template <int BN, int EW, int CTAS = 1> struct Cfg {
  static constexpr int kEpiThreads = EW * 32;
  static constexpr int kThreads = 64 + kEpiThreads;
  static constexpr int kOutBufs = 2;                            // staging tiles per epilogue warp (double buffered)
  static constexpr int kOutBufBytes = (EW == 16) ? 2048 : 4096; // 32 rows x 64 B (16 warps: 32-column bf16 chunks) or 32 rows x 128 B
  static constexpr int kStages = CTAS == 2 ? ((BN == 256) ? 4 : 6) : ((BN == 256) ? 3 : (BN == 128 ? 4 : 6));
  static constexpr int kABytes = BLOCK_M * BLOCK_K * 2;
  static constexpr int kBBytes = (BN / CTAS) * BLOCK_K * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kTmemCols = (2 * BN <= 32) ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
  static constexpr int kStageOutBytes = EW * kOutBufs * kOutBufBytes;   // staging tiles for the TMA stores
  static_assert(kStageBytes % 1024 == 0, "stage alignment");
  static constexpr int kSmemBytes = kStages * kStageBytes + kStageOutBytes + 1024 /*align slack*/ + 256 /*barriers*/ + 4 * BN * 4 /*bias+gamma x2 stages*/;
};

// 16-bit outputs: bf16, or IEEE half (the decoder prefill path) clamped to the finite range first
template <bool F16> __device__ __forceinline__ uint32_t pack2_16(float a, float b) { return F16 ? pack_f16x2_sat(a, b) : pack_bf16x2(a, b); }

struct EpiArgs {
  void* D; int64_t ldd; const float* bias; const float* aux0; int period; int epilogue;
  int dbg;   // developer build only (MDC_GEMM_DBG): 1 = no epilogue body, 2 = every load from tile (0,0), 4 = no loads, 8 = no MMAs, 16 = no output stores, 32 = no TMEM reads
};
#ifdef MDC_DEVTOOLS
#define GEMM_DBG(ep, bit) ((ep).dbg & (bit))
#else
#define GEMM_DBG(ep, bit) 0
#endif

// exact-erf GELU of two values, branch-free:  GELU(x) = x Phi(x) = max(x, 0) - a Phi(-a),  a = |x|,  and  Phi(-a) = 2^q(a)  with q a
// degree-6 polynomial fitted to log2 Phi(-a) on [0, 6] (weighted minimax on the error of a 2^q(a); tools/gelu_fit.py).  |error| of
// GELU <= 2.9e-7 for every x (float32 rounding level at |x| ~ 4; relative error <= 1e-5 down to x -> 0, because the error term carries
// the factor a) -- the same accuracy as the Abramowitz-Stegun 7.1.28 form it replaces (1 - 1/(1+a1 z+...+a6 z^6)^16, 3e-7 on erf), at
// 7 instead of 15 operations on the FP32 pipe per value: the mlp.fc1 epilogue alone took 27 us of a 33 us launch (dev switch
// MDC_GEMM_DBG=12).  a is clamped to 6: beyond it a Phi(-a) < 6e-9.  One MUFU (ex2) per value.
__device__ __forceinline__ void gelu2(uint64_t x, float& y0, float& y1) {
  float x0, x1; upk2(x, x0, x1);
  const float a0 = fminf(fabsf(x0), 6.0f), a1 = fminf(fabsf(x1), 6.0f);
  const uint64_t a = pk2(a0, a1);
  uint64_t p = fma2(a, pk2(3.309269595774822e-05f, 3.309269595774822e-05f), pk2(-0.000769218779169023f, -0.000769218779169023f));
  p = fma2(p, a, pk2(0.008080713450908661f, 0.008080713450908661f));
  p = fma2(p, a, pk2(-0.05341210216283798f, -0.05341210216283798f));
  p = fma2(p, a, pk2(-0.4587709903717041f, -0.4587709903717041f));
  p = fma2(p, a, pk2(-1.1512017250061035f, -1.1512017250061035f));
  p = fma2(p, a, pk2(-0.999993085861206f, -0.999993085861206f));
  float p0, p1; upk2(p, p0, p1);
  y0 = fmaf(-a0, ex2_approx(p0), fmaxf(x0, 0.f));
  y1 = fmaf(-a1, ex2_approx(p1), fmaxf(x1, 0.f));
}

// F16: A, W and the 16-bit outputs are IEEE half instead of bf16 (same bytes, same tensor-core rate, 11 significant bits: the
// decoder's teacher-forced prefill runs on the fp16 decode-loop weights -- DESIGN.md precision policy)
template <int BN, int EPI, int EW, bool F16 = false, int CTAS = 1>
__global__ void __launch_bounds__(64 + EW * 32, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_d,
               EpiArgs ep, int M, int N, int K) {
  using C = Cfg<BN, EW, CTAS>;
  constexpr int EPI_THREADS = C::kEpiThreads;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + C::kStages * C::kABytes;
  uint8_t* smem_out = smem + C::kStages * C::kStageBytes;                 // 1024-aligned (stage sizes are multiples of 1024)
  uint64_t* bars = (uint64_t*)(smem_out + C::kStageOutBytes);
  uint64_t* full = bars;                         // [kStages]
  uint64_t* empty = bars + C::kStages;           // [kStages]
  uint64_t* tmem_full = bars + 2 * C::kStages;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;          // [2]
  uint32_t* tmem_ptr_smem = (uint32_t*)(tmem_empty + 2);
  float* s_bias = (float*)(smem_out + C::kStageOutBytes + 256);          // [2][BN]
  float* s_gamma = s_bias + 2 * BN;                                      // [2][BN]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // a "tile" is 128*CTAS rows x BN columns, owned by a cluster of CTAS CTAs; this CTA computes rows [128*rank, +128) of it
  const uint32_t rank = CTAS == 2 ? cluster_rank() : 0u;
  const int first_tile = blockIdx.x / CTAS, tile_step = gridDim.x / CTAS;
  const int tiles_n = (N + BN - 1) / BN, tiles_m = (M + BLOCK_M * CTAS - 1) / (BLOCK_M * CTAS);
  const int num_tiles = tiles_m * tiles_n;
  const int num_kb = (K + BLOCK_K - 1) / BLOCK_K;

  if (warp == 0 && elect_one()) {
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_w);
    if (EPI != MDC_EPI_PATCH) prefetch_tmap(&map_d);
    for (int i = 0; i < C::kStages; ++i) { mbar_init(smem_u32(&full[i]), 1); mbar_init(smem_u32(&empty[i]), 1); }
    // the accumulator is released by one arrival per epilogue warp of every CTA of the cluster (the leader's barrier is the one waited on)
    for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(&tmem_full[i]), 1); mbar_init(smem_u32(&tmem_empty[i]), EW * CTAS); }
    fence_mbarrier_init();
  } else if (warp == 1) {
    tmem_alloc<CTAS>(smem_u32(tmem_ptr_smem), C::kTmemCols);
    tmem_relinquish<CTAS>();
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CTAS == 2) cluster_sync();      // the peer's barriers are initialised before anything can signal them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===== TMA producer =====
    if (elect_one()) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = first_tile; tile < num_tiles; tile += tile_step) {
        const int m0 = (tile / tiles_n) * (BLOCK_M * CTAS) + rank * BLOCK_M, n0 = (tile % tiles_n) * BN + rank * (BN / CTAS);
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait_spin(smem_u32(&empty[stage]), phase ^ 1);
          const uint32_t fb = smem_u32(&full[stage]);
          if (GEMM_DBG(ep, 4)) { if (rank == 0) mbar_arrive(fb); }
          else if constexpr (CTAS == 2) {
            // both CTAs' loads complete on the LEADER's barrier, which expects the bytes of both
            if (rank == 0) mbar_expect_tx(fb, 2 * C::kStageBytes);
            const uint32_t lb = mapa(fb, 0);
            tma_load_2d_2sm(&map_a, lb, smem_u32(smem_a + stage * C::kABytes), GEMM_DBG(ep, 2) ? 0 : kb * BLOCK_K, GEMM_DBG(ep, 2) ? 0 : m0);
            tma_load_2d_2sm(&map_w, lb, smem_u32(smem_b + stage * C::kBBytes), GEMM_DBG(ep, 2) ? 0 : kb * BLOCK_K, GEMM_DBG(ep, 2) ? 0 : n0);
          } else {
          mbar_expect_tx(fb, C::kStageBytes);
          tma_load_2d(&map_a, fb, smem_u32(smem_a + stage * C::kABytes), GEMM_DBG(ep, 2) ? 0 : kb * BLOCK_K, GEMM_DBG(ep, 2) ? 0 : m0);
          tma_load_2d(&map_w, fb, smem_u32(smem_b + stage * C::kBBytes), GEMM_DBG(ep, 2) ? 0 : kb * BLOCK_K, GEMM_DBG(ep, 2) ? 0 : n0);
          }
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    constexpr uint32_t idesc = make_idesc(BLOCK_M * CTAS, BN, F16);
    int stage = 0; uint32_t phase = 0; int iter = 0;
    if (rank == 0)                                   // the leader CTA of a pair issues for both
    for (int tile = first_tile; tile < num_tiles; tile += tile_step, ++iter) {
      const int as = iter & 1; const uint32_t aphase = (iter >> 1) & 1;
      mbar_wait_spin(smem_u32(&tmem_empty[as]), aphase ^ 1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + as * BN;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait_spin(smem_u32(&full[stage]), phase);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t adesc = make_sw128_desc(smem_u32(smem_a + stage * C::kABytes));
          const uint64_t bdesc = make_sw128_desc(smem_u32(smem_b + stage * C::kBBytes));
          if (!GEMM_DBG(ep, 8))
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) { // +32 B per UMMA_K inside the swizzle atom -> +2 in the >>4 address field
            if constexpr (CTAS == 2) umma_ss_2sm(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
            else umma_ss(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
          }
          if constexpr (CTAS == 2) {
            umma_commit_2sm(smem_u32(&empty[stage]));                       // frees the smem slot in both CTAs when these MMAs retire
            if (kb == num_kb - 1) umma_commit_2sm(smem_u32(&tmem_full[as])); // accumulator ready for both CTAs' epilogues
          } else {
            umma_commit(smem_u32(&empty[stage]));                       // frees the smem slot when these MMAs retire
            if (kb == num_kb - 1) umma_commit(smem_u32(&tmem_full[as])); // accumulator ready for the epilogue
          }
        }
        __syncwarp();
        if (++stage == C::kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ===== epilogue: warp w may only touch TMEM lanes [32*(w%4), +32); warps w and w+4 split the columns =====
    const int quad = warp & 3, half = (warp - 2) >> 2, et = threadIdx.x - 64;     // `half`: which column part of the tile (0 .. EW/4-1)
    constexpr int HALF_COLS = BN / (EW / 4);
    static_assert(HALF_COLS >= 32, "an epilogue warp owns at least 32 columns");
    constexpr bool OUT_F32 = (EPI == MDC_EPI_LS_RESIDUAL);
    // columns per staged chunk: one 32-row x 128-byte tile when the tile half is wide enough, else 32 columns
    static_assert(!(OUT_F32 && EW == 16), "16 epilogue warps: bf16 outputs only (2 KB staging tiles)");
    constexpr int CH = OUT_F32 ? 32 : ((HALF_COLS >= 64 && EW == 8) ? 64 : 32);
    constexpr int ROWB = CH * (OUT_F32 ? 4 : 2);                 // bytes per staged row: 128 (SWIZZLE_128B) or 64 (SWIZZLE_64B)
    const uint32_t stage_out = smem_u32(smem_out) + (warp - 2) * (C::kOutBufs * C::kOutBufBytes);
    int obuf = 0;
    int iter = 0;
    for (int tile = first_tile; tile < num_tiles; tile += tile_step, ++iter) {
      const int as = iter & 1; const uint32_t aphase = (iter >> 1) & 1;
      const int m0 = (tile / tiles_n) * (BLOCK_M * CTAS) + rank * BLOCK_M, n0 = (tile % tiles_n) * BN;
      // stage this tile's bias (and LayerScale gamma) once; overlaps the wait for the accumulator
      for (int i = et; i < BN; i += EPI_THREADS) {
        const bool ok = n0 + i < N;
        s_bias[as * BN + i] = (ok && ep.bias) ? __ldg(ep.bias + n0 + i) : 0.f;
        if (EPI == MDC_EPI_LS_RESIDUAL) s_gamma[as * BN + i] = ok ? __ldg(ep.aux0 + n0 + i) : 0.f;
      }
      bar_sync<1, EPI_THREADS>();
      mbar_wait_spin(smem_u32(&tmem_full[as]), aphase);
      tc_fence_after();
      const int row0 = m0 + quad * 32, row = row0 + lane;
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + as * BN + half * HALF_COLS;
      const float* sb = s_bias + as * BN + half * HALF_COLS;
      const float* sg = s_gamma + as * BN + half * HALF_COLS;
      if (GEMM_DBG(ep, 1)) {
      } else if constexpr (EPI == MDC_EPI_PATCH) {
        // rows are re-mapped past each image's cls slot, so a 32-row box is not contiguous in the output (no TMA store).  The chunk goes
        // through the warp's swizzled staging tile and leaves it in ROW-COALESCED order: eight lanes cover the 128 bytes of a row (four
        // rows per instruction) for the positional-table load and the store -- the thread-per-row form touched 32 lines per instruction
        // and made this epilogue three times the main loop (35 us for a 10 GFLOP GEMM).
        const uint32_t stage_out = smem_u32(smem_out) + (warp - 2) * (C::kOutBufs * C::kOutBufBytes);
        static_assert(C::kOutBufBytes >= 4096, "one 32-row x 128-byte staging tile per epilogue warp");
#pragma unroll 1
        for (int c0 = 0; c0 < HALF_COLS; c0 += 32) {
          const int col0 = n0 + half * HALF_COLS + c0;
          uint32_t v[32];
          tmem_ld32(taddr + c0, v);
          tmem_ld_wait();
          const uint32_t row_s = stage_out + lane * 128;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b4 = *reinterpret_cast<const float4*>(sb + c0 + 4 * j);
            sts128(row_s + ((j ^ (lane & 7)) << 4), __float_as_uint(__uint_as_float(v[4 * j]) + b4.x), __float_as_uint(__uint_as_float(v[4 * j + 1]) + b4.y),
                   __float_as_uint(__uint_as_float(v[4 * j + 2]) + b4.z), __float_as_uint(__uint_as_float(v[4 * j + 3]) + b4.w));
          }
          __syncwarp();
          const int ch = lane & 7, col = col0 + 4 * ch;
          const int img0 = row0 / ep.period;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rl = i * 4 + (lane >> 3), r = row0 + rl;
            const uint4 xu = lds128(stage_out + rl * 128 + ((ch ^ (rl & 7)) << 4));
            const float4 x = make_float4(__uint_as_float(xu.x), __uint_as_float(xu.y), __uint_as_float(xu.z), __uint_as_float(xu.w));
            if (r < M && col < N) {
              int img = img0, pr = r - img0 * ep.period;
              if (pr >= ep.period) { pr -= ep.period; ++img; }                     // a 32-row chunk crosses at most one image boundary
              const float4 pz = __ldg(reinterpret_cast<const float4*>(ep.aux0 + (int64_t)pr * ep.ldd + col));
              *reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.D) + (int64_t)(r + img + 1) * ep.ldd + col) =
                  make_float4(x.x + pz.x, x.y + pz.y, x.z + pz.z, x.w + pz.w);
            }
          }
          __syncwarp();
        }
      } else {
        // TMEM -> registers -> epilogue math -> swizzled staging tile in shared memory -> one TMA store (bf16 outputs) or TMA
        // reduce-add into the fp32 residual stream (LayerScale + residual: R += gamma * (acc + bias), added exactly once per
        // element, so the result equals the read-modify-write) per 32-row x CH-column chunk.  No per-thread global access.
#pragma unroll 1
        for (int c0 = 0; c0 < HALF_COLS; c0 += CH) {
          const int col0 = n0 + half * HALF_COLS + c0;
          uint32_t v[CH];
          if (GEMM_DBG(ep, 32)) {
#pragma unroll
            for (int i = 0; i < CH; ++i) v[i] = 0x3f800000u + lane + i;
          } else {
          tmem_ld32(taddr + c0, v);
          if constexpr (CH == 64) tmem_ld32(taddr + c0 + 32, v + 32);
          }
          if (lane == 0) bulk_wait_read<C::kOutBufs - 1>();   // the store last issued from this staging buffer has read it
          __syncwarp();
          tmem_ld_wait();
          const uint32_t tile_s = stage_out + obuf * C::kOutBufBytes;
          const uint32_t row_s = tile_s + lane * ROWB;
#pragma unroll
          for (int j = 0; j < CH; j += 8) {               // 8 columns -> one 16-byte chunk (bf16) or two (fp32)
            float o[8];
            const float4 b0 = *reinterpret_cast<const float4*>(sb + c0 + j), b1 = *reinterpret_cast<const float4*>(sb + c0 + j + 4);
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int jj = 0; jj < 8; jj += 2) {
              if constexpr (EPI == MDC_EPI_BIAS_GELU) {
                gelu2(add2(pk2(__uint_as_float(v[j + jj]), __uint_as_float(v[j + jj + 1])), pk2(bb[jj], bb[jj + 1])), o[jj], o[jj + 1]);
              } else {
                float a0 = __uint_as_float(v[j + jj]) + bb[jj], a1 = __uint_as_float(v[j + jj + 1]) + bb[jj + 1];
                if (EPI == MDC_EPI_BIAS_RELU) { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); }
                o[jj] = a0; o[jj + 1] = a1;
              }
            }
            if constexpr (OUT_F32) {
              const float4 g0 = *reinterpret_cast<const float4*>(sg + c0 + j), g1 = *reinterpret_cast<const float4*>(sg + c0 + j + 4);
              const int c = j >> 2;                        // 16-byte chunk index within the 128-byte row
              sts128(row_s + (((c) ^ (lane & 7)) << 4), __float_as_uint(o[0] * g0.x), __float_as_uint(o[1] * g0.y), __float_as_uint(o[2] * g0.z), __float_as_uint(o[3] * g0.w));
              sts128(row_s + (((c + 1) ^ (lane & 7)) << 4), __float_as_uint(o[4] * g1.x), __float_as_uint(o[5] * g1.y), __float_as_uint(o[6] * g1.z), __float_as_uint(o[7] * g1.w));
            } else {
              const int c = j >> 3;
              const int sw = (ROWB == 128) ? (lane & 7) : ((lane >> 1) & 3);
              sts128(row_s + ((c ^ sw) << 4), pack2_16<F16>(o[0], o[1]), pack2_16<F16>(o[2], o[3]), pack2_16<F16>(o[4], o[5]), pack2_16<F16>(o[6], o[7]));
            }
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0 && row0 < M && col0 < N && !GEMM_DBG(ep, 16)) {
            const int sc = GEMM_DBG(ep, 64) ? 0 : col0, sr = GEMM_DBG(ep, 64) ? 0 : row0;      // 64: every store to tile (0,0)
            if constexpr (OUT_F32) tma_reduce_add_2d(&map_d, tile_s, sc, sr);
            else tma_store_2d(&map_d, tile_s, sc, sr);
          }
          if (lane == 0) bulk_commit();
          if (C::kOutBufs == 2) obuf ^= 1;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {                                            // this warp's TMEM reads of the accumulator stage are done
        if constexpr (CTAS == 2) mbar_arrive_cluster(smem_u32(&tmem_empty[as]), 0);
        else mbar_arrive(smem_u32(&tmem_empty[as]));
      }
    }
    if (EPI != MDC_EPI_PATCH && lane == 0) bulk_wait_read<0>();   // staging tiles must outlive the last stores' reads
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CTAS == 2) cluster_sync();      // no CTA leaves while its peer can still signal its barriers or read its operands
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<CTAS>(tmem_base, C::kTmemCols);
  }
}

// ---- host side: tensor-map cache --------------------------------------------------------------------
struct TmapKey {
  const void* ptr; int64_t rows, cols, ld; int box_rows;
  bool operator==(const TmapKey& o) const { return ptr == o.ptr && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows; }
};
struct TmapHash {
  size_t operator()(const TmapKey& k) const {
    size_t h = (size_t)k.ptr; h ^= (size_t)k.rows * 0x9E3779B97F4A7C15ull; h ^= (size_t)k.cols * 0xC2B2AE3D27D4EB4Full;
    h ^= (size_t)k.ld * 0x165667B19E3779F9ull; h ^= (size_t)k.box_rows << 7; return h;
  }
};
struct TmapCache { std::unordered_map<TmapKey, CUtensorMap, TmapHash> map; std::mutex mu; };

int get_tmap(mdc_ctx* ctx, const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows, CUtensorMap* out) {
  if (!ctx->encode_fn) {
    void* fn = nullptr; cudaDriverEntryPointQueryResult qres;
    MDC_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || !fn) MDC_FAIL(-3, "cuTensorMapEncodeTiled entry point unavailable");
    ctx->encode_fn = fn;
  }
  if (!ctx->tmap_cache) ctx->tmap_cache = new TmapCache();
  TmapCache* c = (TmapCache*)ctx->tmap_cache;
  TmapKey key{ptr, rows, cols, ld, box_rows};
  std::lock_guard<std::mutex> lk(c->mu);
  auto it = c->map.find(key);
  if (it != c->map.end()) { *out = it->second; return 0; }
  auto encode = (PFN_cuTensorMapEncodeTiled_v12000)ctx->encode_fn;
  CUtensorMap m;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) MDC_FAIL(-3, "cuTensorMapEncodeTiled failed (%d) ptr=%p rows=%lld cols=%lld ld=%lld", (int)r, ptr, (long long)rows, (long long)cols, (long long)ld);
  if (c->map.size() > 4096) c->map.clear();
  c->map.emplace(key, m);
  *out = m; return 0;
}

// tensor map of the output for the epilogue's TMA stores: box = 32 rows x `box_cols` columns (128 or 64 bytes per row)
int make_out_tmap(mdc_ctx* ctx, const void* ptr, int64_t rows, int64_t cols, int64_t ld, bool f32, int box_cols, CUtensorMap* out) {
  auto encode = (PFN_cuTensorMapEncodeTiled_v12000)ctx->encode_fn;
  const int es = f32 ? 4 : 2;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * es};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, 32u};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw = (box_cols * es == 128) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = encode(out, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) MDC_FAIL(-3, "cuTensorMapEncodeTiled (output) failed (%d) ptr=%p rows=%lld cols=%lld ld=%lld", (int)r, ptr, (long long)rows, (long long)cols, (long long)ld);
  return 0;
}

template <int BN, int EPI, bool F16 = false, int CTAS = 1>
int launch_bn_epi(mdc_ctx* ctx, const CUtensorMap& ma, const CUtensorMap& mw, const EpiArgs& ep, int M, int N, int K, cudaStream_t s) {
  constexpr int EW = (BN == 256 && EPI == MDC_EPI_BIAS_GELU) ? 16 : 8;     // A/B on one box: fc1 34.0 -> 31.6 us; bias-only epilogues lose 3 %
  using C = Cfg<BN, EW, CTAS>;
  static bool attr_set[MDC_MAX_DEVICES];      // the dynamic-smem opt-in is a per-device attribute of this instantiation
  if (ctx->device < 0 || ctx->device >= MDC_MAX_DEVICES) MDC_FAIL(-2, "device index %d out of range", ctx->device);
  if (!attr_set[ctx->device]) {
    MDC_CUDA(cudaFuncSetAttribute(gemm_tc_kernel<BN, EPI, EW, F16, CTAS>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes));
    attr_set[ctx->device] = true;
  }
  const int tiles = ((M + BLOCK_M * CTAS - 1) / (BLOCK_M * CTAS)) * ((N + BN - 1) / BN);     // tiles of 128*CTAS rows, one cluster each
  int max_clusters = ctx->sm_count / CTAS;
#ifdef MDC_DEVTOOLS
  if (const char* e = getenv("MDC_GEMM_GRID")) { const int g = atoi(e) / CTAS; if (g >= 1 && g < max_clusters) max_clusters = g; }
#endif
  const int grid = (tiles < max_clusters ? tiles : max_clusters) * CTAS;
  CUtensorMap md;
  memset(&md, 0, sizeof(md));
  if (EPI != MDC_EPI_PATCH) {
    const bool f32 = (EPI == MDC_EPI_LS_RESIDUAL);
    const int box_cols = f32 ? 32 : ((BN / (EW / 4) >= 64 && EW == 8) ? 64 : 32);
    MDC_TRY(make_out_tmap(ctx, ep.D, M, N, ep.ldd, f32, box_cols, &md));
  }
  if constexpr (CTAS == 1) {
    gemm_tc_kernel<BN, EPI, EW, F16, 1><<<grid, C::kThreads, C::kSmemBytes, s>>>(ma, mw, md, ep, M, N, K);
  } else {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(C::kThreads); cfg.dynamicSmemBytes = C::kSmemBytes; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = CTAS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    MDC_CUDA(cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, EPI, EW, F16, CTAS>, ma, mw, md, ep, M, N, K));
  }
  MDC_LAUNCH_CHECK(ctx);
  return 0;
}

template <int BN, int CTAS = 1>
int launch_bn(mdc_ctx* ctx, const CUtensorMap& ma, const CUtensorMap& mw, const EpiArgs& ep, int M, int N, int K, cudaStream_t s) {
  switch (ep.epilogue) {
    case MDC_EPI_BIAS: return launch_bn_epi<BN, MDC_EPI_BIAS, false, CTAS>(ctx, ma, mw, ep, M, N, K, s);
    case MDC_EPI_BIAS_GELU: return launch_bn_epi<BN, MDC_EPI_BIAS_GELU, false, CTAS>(ctx, ma, mw, ep, M, N, K, s);
    case MDC_EPI_BIAS_RELU: return launch_bn_epi<BN, MDC_EPI_BIAS_RELU, false, CTAS>(ctx, ma, mw, ep, M, N, K, s);
    case MDC_EPI_LS_RESIDUAL: return launch_bn_epi<BN, MDC_EPI_LS_RESIDUAL, false, CTAS>(ctx, ma, mw, ep, M, N, K, s);
    case MDC_EPI_PATCH: return launch_bn_epi<BN, MDC_EPI_PATCH, false, 1>(ctx, ma, mw, ep, M, N, K, s);     // direct-store epilogue: single-CTA tiles only
  }
  MDC_FAIL(-2, "gemm: unknown epilogue %d", ep.epilogue);
}

template <int BN>
int launch_bn_f16(mdc_ctx* ctx, const CUtensorMap& ma, const CUtensorMap& mw, const EpiArgs& ep, int M, int N, int K, cudaStream_t s) {
  switch (ep.epilogue) {       // the epilogues the decoder prefill uses
    case MDC_EPI_BIAS: return launch_bn_epi<BN, MDC_EPI_BIAS, true>(ctx, ma, mw, ep, M, N, K, s);
    case MDC_EPI_BIAS_RELU: return launch_bn_epi<BN, MDC_EPI_BIAS_RELU, true>(ctx, ma, mw, ep, M, N, K, s);
  }
  MDC_FAIL(-2, "gemm (fp16 operands): epilogue %d is not available, only MDC_EPI_BIAS / MDC_EPI_BIAS_RELU", ep.epilogue);
}

}  // namespace

int gemm_tc_supported(int M, int N, int K, int64_t lda, int64_t ldw) {
  // TMA: 16-byte aligned row pitch; epilogue vector paths want N % 8 == 0
  return (K % 8 == 0) && (lda % 8 == 0) && (ldw % 8 == 0) && (N % 8 == 0) && M >= 1;
}

int gemm_tc_launch(mdc_ctx* ctx, int epilogue, const void* A, int64_t lda, const void* W, int64_t ldw, void* D, int64_t ldd,
                   const float* bias, const float* aux0, int period, int M, int N, int K, cudaStream_t s, int f16) {
  MDC_CHECK_ARG(((uintptr_t)A & 15) == 0 && ((uintptr_t)W & 15) == 0 && ((uintptr_t)D & 15) == 0);
  MDC_CHECK_ARG(ldd % 8 == 0);
  if (epilogue == MDC_EPI_PATCH) MDC_CHECK_ARG(period >= 32);      // a 32-row epilogue chunk crosses at most one image boundary
  if (epilogue == MDC_EPI_PATCH) MDC_CHECK_ARG(((uintptr_t)aux0 & 15) == 0);   // the positional rows are read as float4
  // tile width: the widest tile that still gives every SM one tile (128 x 256 tiles need 1/3 less operand traffic per flop than
  // 128 x 128 ones; with N = 512 that is 1.3 waves instead of 2.7 -- the same time for the kernel alone, ~1 % more images/s in the
  // batch pipeline, where co-scheduled kernels fill the tail and SM-time is what counts); narrow N uses narrow tiles
  const int tiles_m = (M + BLOCK_M - 1) / BLOCK_M;
  int bn = 128;
  if (N % 256 == 0 && tiles_m * (N / 256) >= ctx->sm_count) bn = 256;
  if (N <= 64 || tiles_m * ((N + 127) / 128) < ctx->sm_count) bn = 64;
  // CTA pairs (cta_group::2) for the wide tiles of tall problems: a third less shared-memory traffic per flop
  int ctas = (!f16 && bn >= 128 && epilogue != MDC_EPI_PATCH && M >= 2 * BLOCK_M) ? 2 : 1;
#ifdef MDC_DEVTOOLS
  if (const char* e = getenv("MDC_GEMM_2CTA")) ctas = (e[0] == '0') ? 1 : ctas;
#endif
  CUtensorMap ma, mw;
  MDC_TRY(get_tmap(ctx, A, M, K, lda, BLOCK_M, &ma));
  MDC_TRY(get_tmap(ctx, W, N, K, ldw, bn / ctas, &mw));        // a CTA of a pair loads half of the B tile
  EpiArgs ep{D, ldd, bias, aux0, period, epilogue, 0};
#ifdef MDC_DEVTOOLS
  if (const char* e = getenv("MDC_GEMM_DBG")) ep.dbg = atoi(e);
#endif
  if (f16) {
    if (bn == 256) return launch_bn_f16<256>(ctx, ma, mw, ep, M, N, K, s);
    if (bn == 128) return launch_bn_f16<128>(ctx, ma, mw, ep, M, N, K, s);
    return launch_bn_f16<64>(ctx, ma, mw, ep, M, N, K, s);
  }
  if (ctas == 2) return bn == 256 ? launch_bn<256, 2>(ctx, ma, mw, ep, M, N, K, s) : launch_bn<128, 2>(ctx, ma, mw, ep, M, N, K, s);
  if (bn == 256) return launch_bn<256>(ctx, ma, mw, ep, M, N, K, s);
  if (bn == 128) return launch_bn<128>(ctx, ma, mw, ep, M, N, K, s);
  return launch_bn<64>(ctx, ma, mw, ep, M, N, K, s);
}

// Generic 2-D bf16 tensor map (used by the cluster decode kernel): tensor [rows, cols] with row pitch `ld` elements,
// box [box_cols, box_rows]; swizzle_mode 0 = none, 1 = 32B, 2 = 64B, 3 = 128B (box_cols * 2 bytes must not exceed the swizzle span).
int mdc_make_tmap_2d(mdc_ctx* ctx, const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows, int swizzle_mode, void* out_map) {
  if (!ctx->encode_fn) {
    void* fn = nullptr; cudaDriverEntryPointQueryResult qres;
    MDC_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || !fn) MDC_FAIL(-3, "cuTensorMapEncodeTiled entry point unavailable");
    ctx->encode_fn = fn;
  }
  auto encode = (PFN_cuTensorMapEncodeTiled_v12000)ctx->encode_fn;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw = swizzle_mode == 3 ? CU_TENSOR_MAP_SWIZZLE_128B : swizzle_mode == 2 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle_mode == 1 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = encode((CUtensorMap*)out_map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) MDC_FAIL(-3, "cuTensorMapEncodeTiled failed (%d) ptr=%p rows=%lld cols=%lld ld=%lld box=%dx%d", (int)r, ptr,
                                  (long long)rows, (long long)cols, (long long)ld, box_cols, box_rows);
  return 0;
}

void gemm_tc_ctx_destroy(mdc_ctx* ctx) {
  if (ctx && ctx->tmap_cache) { delete (TmapCache*)ctx->tmap_cache; ctx->tmap_cache = nullptr; }
}
