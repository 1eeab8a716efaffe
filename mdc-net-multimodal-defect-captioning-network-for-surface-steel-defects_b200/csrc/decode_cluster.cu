// decode_cluster.cu -- the whole autoregressive decode loop as ONE persistent, cluster-cooperative kernel
// (north_star (c)+(d): paged bf16 self-KV, L2/HBM-resident cross-K/V, LayerNorm + residual + token select fused;
//  "no collective inside the decode loop" -- here not even a kernel boundary).
//
// Decomposition (model width 256, 8 heads x 32, FFN 2048 -- the configuration inference_p.py:126-129 builds):
//   * a thread-block CLUSTER of 8 CTAs owns a group of G <= 8 images (G <= 16 in the two-column-block instantiation the
//     batch pipeline uses) for the entire loop; clusters never talk to each other, so there is no grid-wide
//     synchronisation at all.  Further groups are processed back to back.
//   * inside a cluster CTA r owns attention head r and 1/8 of every projection: in-proj rows of head r (q,k,v),
//     out-proj / cross-q / cross-out rows [32r,32r+32), FFN1 hidden units [256r,256r+256), FFN2 as a K-split over
//     the same hidden units, vocabulary rows [40r,40r+40).
//   * everything that is read from HBM/L2 -- weights, the paged self-KV cache, the resident cross-K/V -- is fetched
//     by a dedicated PRODUCER WARP with TMA (cp.async.bulk.tensor, hardware 128B/64B swizzle) into a 5 x 32 KB (4 x 32 KB
//     with 16 images) shared-memory ring guarded by full/empty mbarriers; the producer walks the static stage schedule and runs
//     ahead of the 8 consumer warps across phase, layer and step boundaries.
//   * projections run on the tensor cores with the roles swapped: the WEIGHT rows are the MMA M dimension
//     (mma.sync m16n8k16, A fragments by ldmatrix from the swizzled TMA tile), the images are the N = 8
//     dimension (one or two column blocks per weight fragment), so no MMA lane is wasted on padding.  The decode-loop weights are IEEE fp16 (the weight table of mdc_b200.h: same
//     bytes as bf16, 8x smaller rounding) and so are the projection operands (activations rounded to fp16: 11 significant bits).
//     Attention keeps bf16 K/V (the caches) with bf16 queries and probabilities.
//   * activations (a few KB) are exchanged through DISTRIBUTED SHARED MEMORY, push style: the producer of a slice
//     writes it into every peer with st.async (...mbarrier::complete_tx), the consumer waits on a local mbarrier
//     for the expected byte count.  No cluster-wide barrier inside the loop.
//   * LayerNorm+residual are fused into the all-gathers; the head's logits go straight to the CTA that owns the
//     image, which runs the greedy / top-k / top-p select and broadcasts the token.
// The generic kernels in decode.cu remain the path for the fp32 token-exact mode and other geometries;
// mdc_decode_steps picks this kernel when the geometry matches.
#include "common.cuh"
#include <cuda_fp16.h>
#include <stdlib.h>
#include <string.h>

#define MDC_SEL_SYNC() bar_sync<1, 256>()
#include "select.cuh"
using namespace mdcsel;

namespace {

constexpr int CS = 8;              // cluster size == heads
constexpr int DM = 256;            // model width
constexpr int HD = 32;             // head width
constexpr int FFN = 2048;
constexpr int FS = FFN / CS;       // hidden units per CTA (256)
constexpr int NCT = 256;           // consumer threads (8 warps)
constexpr int NT = NCT + 32;       // + producer warp
constexpr int XP = DM + 8;         // fp16 elements per padded activation row (528 B: conflict-free ldmatrix)
constexpr int BLK_BYTES = 16384;     // one 32-row weight block (32 rows x 512 B); a ring stage holds NB of them, or one 16-key chunk of every image's K and V
constexpr int VSL = 40;            // vocab rows per CTA; 8*40 = 320 >= V
constexpr int OSTR = 36;           // floats per image in the attention output staging: o[32], running max, softmax denominator, -, -
constexpr int NS_MAX = 10;

// ---- shared memory map (bytes from the 1024-aligned base), per instantiation -------------------------------------
// NB = 8-image column blocks per cluster pass: NB = 1 (up to 8 images per cluster: lowest latency, the serial path) or NB = 2
// (up to 16 images: every weight fragment a warp loads feeds two MMA column blocks, every exchange carries twice the images and
// every warp attends for two images at a time -- less SM-time per image, used by the batch pipeline).  A ring stage is
// NB x 16 KB: NB weight blocks of 32 rows, or one 16-key chunk of the K and V head slices of all 8 NB images.
// OVL: the select scratch shares its bytes with the q/k/v/y staging (disjoint phases); always on with NB = 2, with NB = 1 it
// makes the two-CTAs-per-SM layout fit.
template <int NB, int NSTG, bool OVL>
struct Lay {
  static constexpr int GMX = 8 * NB;                             // max images per cluster pass
  static constexpr int NS = NSTG;                                // ring stages
  static constexpr int STAGE = NB * BLK_BYTES;
  static constexpr int ACT_BYTES = GMX * XP * 2;
  static constexpr int OFF_RING = 0;
  static constexpr int OFF_XH = OFF_RING + NS * STAGE;            // LN output (fp16 projection operand)
  static constexpr int OFF_OH = OFF_XH + ACT_BYTES;               // gathered attention output (written by peers)
  static constexpr int OFF_FH = OFF_OH + ACT_BYTES;               // own FFN hidden slice
  static constexpr int OFF_XRES = OFF_FH + ACT_BYTES;             // [GMX][DM] f32 residual stream
  static constexpr int OFF_YRECV = OFF_XRES + GMX * DM * 4;       // [GMX][DM] f32 all-gathered projection output (peers write)
  static constexpr int F2_BYTES = CS * GMX * 32 * 4;              // [CS src][GMX][32] f32 FFN2 partial sums (peers write)
  static constexpr int OFF_F2RECV = OFF_YRECV + GMX * DM * 4;
  static constexpr int OFF_QS = OFF_F2RECV + F2_BYTES;            // [GMX][32] f32 scaled query of the own head
  static constexpr int OFF_KNEW = OFF_QS + GMX * 32 * 4;          // [GMX][32] f32 this step's key (bf16-rounded)
  static constexpr int OFF_VNEW = OFF_KNEW + GMX * 32 * 4;
  static constexpr int OFF_YTMP = OFF_VNEW + GMX * 32 * 4;        // [GMX][32] f32 own slice of a projection before the push
  static constexpr int OFF_OST = OFF_YTMP + GMX * 32 * 4;         // [GMX][OSTR] f32 attention output staging (fragment -> channel order)
  static constexpr int OFF_QH = OFF_OST + GMX * OSTR * 4;         // [GMX][32] bf16 scaled query (MMA A operand)
  static constexpr int OFF_LRECV = OFF_QH + GMX * 32 * 2;         // [NB][CS src][VSL] f32 logits of the images this CTA selects for
  static constexpr int SEL_BYTES = (CS * VSL + 512) * 4;          // select scratch: 320 + 512 floats
  static constexpr int OFF_SEL = !OVL ? OFF_LRECV + NB * CS * VSL * 4 : OFF_QS;
  static constexpr int OFF_TOK = !OVL ? OFF_SEL + SEL_BYTES : OFF_LRECV + NB * CS * VSL * 4;    // [2][GMX] int32 (double buffered by step parity)
  static constexpr int OFF_PAGES = OFF_TOK + 2 * GMX * 4;         // [GMX][32] int32
  static constexpr int OFF_PADF = OFF_PAGES + GMX * 32 * 4;       // [GMX][8] u32: bit u of an image's 256-bit row = token u is PAD
  static constexpr int OFF_HASPAD = OFF_PADF + GMX * 32;          // [GMX] int32: any PAD token among the keys so far
  static constexpr int OFF_FIN = OFF_HASPAD + GMX * 4;            // stop at EOS: [2] u32 finished masks (by step parity), int all-finished,
                                                                  // u32 the producer's BAR_STEP phase
  static constexpr int OFF_BARS = OFF_FIN + 16;                   // mbarriers
  static constexpr int NBARS = 2 * NS_MAX + 6;
  static constexpr int SMEM_USED = OFF_BARS + NBARS * 8;
  static constexpr int SMEM_BYTES = SMEM_USED + 1024;             // + alignment slack
  static constexpr int OFF_PLEN = SMEM_USED;                      // kPrompt only: [GMX] int32 prompt lengths of the group, past the
  static constexpr int SMEM_BYTES_PROMPT = SMEM_BYTES + GMX * 4;  // layout of the instantiations without a prompt (which stays as it was)
  static_assert(SMEM_BYTES_PROMPT <= 227 * 1024, "shared memory budget");
  static_assert(OFF_XH % 16 == 0 && OFF_XRES % 16 == 0 && OFF_F2RECV % 16 == 0 && OFF_QS % 16 == 0 && OFF_OST % 16 == 0 && OFF_BARS % 8 == 0, "alignment");
  static_assert(!OVL || 4 * GMX * 32 * 4 >= SEL_BYTES, "select scratch must fit the q/k/v/y staging it shares");
  static_assert(GMX * 2048 == STAGE, "a 16-key chunk of all images' K and V head slices fills a stage");
};

// BAR_STEP (stop at EOS only): the consumers' decision whether step t runs, handed to the producer before it emits step t's stages
enum { BAR_FULL = 0, BAR_EMPTY = NS_MAX, BAR_O = 2 * NS_MAX, BAR_Y, BAR_F2, BAR_LG, BAR_TOK, BAR_STEP, BAR_COUNT };

constexpr int BLOCKS_PER_LAYER = 22;   // packed weight blocks per (layer, CTA rank): in-proj q,k,v | self out | cross q | cross out | FFN1 x8 | FFN2 x8
constexpr int HEAD_PACK_BYTES = BLK_BYTES + 8 * 512;    // per rank: vocabulary rows [0,32) as a 32-row block + rows [32,40) as an 8-row block

struct __align__(64) FusedParams {
  const uint8_t* wpack;          // packed decode-loop weights (mdc_decode_pack): ready-to-use shared-memory images, one bulk copy per stage
  const uint8_t* ckv_pack;       // packed cross-K/V (mdc_cross_kv_build): [layer][image][head][16-key chunk] x 2 KB
  const float* b_in[8]; const float* b_so[8]; const float* ln1w[8]; const float* ln1b[8];
  const float* b_ca[8]; const float* b_co[8]; const float* ln2w[8]; const float* ln2b[8];
  const float* b_f1[8]; const float* b_f2[8]; const float* ln3w[8]; const float* ln3b[8];
  const float* emb; const float* pos; const float* b_out;
  int layers, vocab, S, pad_idx;
  int B, G, n_groups;
  int32_t* tokens; int tokens_ld;
  bf16* kv_pool; const int32_t* page_table; int pages_per_seq, PT;
  float* logits_out; int64_t logits_img_stride; int logits_row_offset;
  float* confs; int confs_ld;
  const float* uniforms; int uniforms_ld; int top_k; float top_p; int forced;
  int eos;                                 // mdc_decode_state.eos_token (read by the kStop instantiations)
  int t_begin, t_end;
  long long* trace; int trace_t;           // developer aid: phase timestamps of CTA 0 at step trace_t (MDC_DECODE_TRACE_PTR)
  float ref_margin;                        // developer build: softmax reference-maximum margin (MDC_DECODE_REF_MARGIN; the product build uses 64)
  const int32_t* prompt_len;               // mdc_decode_state.prompt_len (read by the kPrompt instantiations)
};

__device__ __forceinline__ void cbar() { bar_sync<1, NCT>(); }   // the 8 consumer warps

// One 16-row tile of a projection with the weights as the M operand:
//   acc[nb][0..3] = D[m0+g][img], D[m0+g][img+1], D[m0+g+8][img], D[m0+g+8][img+1], img = 8nb + 2q   (g = lane/4, q = lane%4)
// wblk: shared address of the TMA row block [4 k-blocks][R rows][128 B] (SWIZZLE_128B), fp16 weights; bh: fp16 activations
// [8 images][XP].  The fragment loads run two iterations ahead of the MMAs (the asm statements are volatile, so program order
// IS issue order: without the explicit skew every iteration pays the full ldmatrix latency; the buffer of iteration i is
// refilled for iteration i+2 as soon as its MMAs are issued); four accumulator chains.
template <int R, int NB>
__device__ __forceinline__ void mma_mtile(uint32_t wblk, int m0, uint32_t bh, float (&acc)[NB][4]) {
  const int lane = threadIdx.x & 31;
  const int row = m0 + (lane & 7) + ((lane >> 3) & 1) * 8, csel = lane >> 4, sw = lane & 7;
  const uint32_t a_base = wblk + row * 128;
  const uint32_t b_base = bh + (lane & 7) * (XP * 2) + (lane >> 3) * 16;
  float c[NB][4][4];
#pragma unroll
  for (int nb = 0; nb < NB; ++nb)
#pragma unroll
    for (int j = 0; j < 4; ++j) { c[nb][j][0] = c[nb][j][1] = c[nb][j][2] = c[nb][j][3] = 0.f; }
  uint32_t a0[2][4], a1[2][4], xb[2][NB][4];
#define MDC_MTILE_LOAD(I)                                                                                      \
  {                                                                                                            \
    constexpr int i_ = (I), kb_ = i_ >> 1, ch_ = (i_ & 1) * 4, buf_ = i_ & 1;                                  \
    ldsm_x4(a0[buf_], a_base + kb_ * (R * 128) + (((ch_ + csel) ^ sw) << 4));                                  \
    ldsm_x4(a1[buf_], a_base + kb_ * (R * 128) + (((ch_ + 2 + csel) ^ sw) << 4));                              \
    _Pragma("unroll") for (int nb_ = 0; nb_ < NB; ++nb_) ldsm_x4(xb[buf_][nb_], b_base + nb_ * (8 * XP * 2) + i_ * 64); \
  }
#define MDC_MTILE_MMA(I)                                                                                       \
  {                                                                                                            \
    constexpr int i_ = (I), buf_ = i_ & 1, par_ = (i_ & 1) * 2;                                                \
    _Pragma("unroll") for (int nb_ = 0; nb_ < NB; ++nb_) {                                                     \
      mma_m16n8k16<__half>(c[nb_][par_], a0[buf_], xb[buf_][nb_][0], xb[buf_][nb_][1]);                        \
      mma_m16n8k16<__half>(c[nb_][par_ + 1], a1[buf_], xb[buf_][nb_][2], xb[buf_][nb_][3]);                    \
    }                                                                                                          \
  }
  MDC_MTILE_LOAD(0) MDC_MTILE_LOAD(1)
  MDC_MTILE_MMA(0) MDC_MTILE_LOAD(2)
  MDC_MTILE_MMA(1) MDC_MTILE_LOAD(3)
  MDC_MTILE_MMA(2) MDC_MTILE_LOAD(4)
  MDC_MTILE_MMA(3) MDC_MTILE_LOAD(5)
  MDC_MTILE_MMA(4) MDC_MTILE_LOAD(6)
  MDC_MTILE_MMA(5) MDC_MTILE_LOAD(7)
  MDC_MTILE_MMA(6) MDC_MTILE_MMA(7)
#undef MDC_MTILE_LOAD
#undef MDC_MTILE_MMA
#pragma unroll
  for (int nb = 0; nb < NB; ++nb)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[nb][j] = (c[nb][0][j] + c[nb][1][j]) + (c[nb][2][j] + c[nb][3][j]);
}

// ---- attention of ONE query per image on the tensor cores ------------------------------------------------------
// A key / value panel in shared memory holds key u at u*64 bytes, 16-byte chunk c stored at c ^ ((u >> 1) & 3)
// (TMA SWIZZLE_64B).  The query (bf16, like the K/V it meets -- the precision of the caches; tools/error_budget_cpu.py: "q bf16",
// "p bf16" move the logit error by < 5e-4) is row 0 of the M operand of S = q.K^T, so the score of keys 2q, 2q+1 of an 8-key
// tile lands in lanes (g = 0, q) -- exactly where the B fragment of P.V wants column 0: the softmax runs in registers, nothing
// goes through shared memory.  Lanes of the other row groups compute on zero rows; their values only reach output columns
// that are never read.  Scores are in log2 units (q is pre-scaled by log2(e)/sqrt(hd)), so p = exp2(s - m).

// A fragments of q from its bf16 row (32 dims): aq[ks][h] covers dims 16*ks + 8*h + {2q, 2q+1}.  The query fills ALL eight row groups
// of the M operand (rows 8-15 stay zero): every row group then computes the same scores, so the running maximum, the rescale factor
// and the probabilities are identical in all lanes of a quad column and every column of P.V carries the output -- no broadcast.
__device__ __forceinline__ void build_q_frag(const bf16* qh, uint32_t (&aq)[2][2]) {
  const int q4 = threadIdx.x & 3;
  const bf16* src = qh + 2 * q4;
#pragma unroll
  for (int i = 0; i < 4; ++i) aq[i >> 1][i & 1] = *reinterpret_cast<const uint32_t*>(src + (i >> 1) * 16 + (i & 1) * 8);
}

// running state of one (image, head) attention job, owned by ONE warp for the whole key range (flash-style online softmax):
// m: running maximum (log2 units), ls: this lane's share of the softmax denominator (lanes of a quad hold different keys),
// o: un-normalised output, dims mt*16 + {g, g+8} as o[mt][0] / o[mt][2] (every lane of the row group holds a copy).
struct AttnState { float m, ls; float o[2][4]; };

// One 16-key tile (a [16 keys][64 B] K panel and V panel, TMA SWIZZLE_64B: 16-byte chunk c of key r at c ^ ((r >> 1) & 3)) for N
// images at once, written phase by phase across the images (the asm statements are volatile: program order is issue order), so
// that the two images of a warp overlap their ldmatrix / MMA / shuffle latencies.  key0: index of the tile's first key; keys
// >= nkeys are masked; padw: PAD bit rows (or null).
template <int N>
__device__ __forceinline__ void attn_tile(const uint32_t (&kp)[N], const uint32_t (&vp)[N], const uint32_t (&aq)[N][2][2], int key0, int nkeys,
                                          const uint32_t* const (&padw)[N], AttnState (&st)[N], float margin) {
  const int lane = threadIdx.x & 31, q4 = lane & 3;
  uint32_t kb[N][2][4], va[N][2][4];
#pragma unroll
  for (int n = 0; n < N; ++n)
#pragma unroll
    for (int j = 0; j < 2; ++j) {              // 8-key n-tile j: one ldmatrix.x4 = the four dim chunks of keys 8j .. 8j+7
      const int r = 8 * j + (lane & 7);
      ldsm_x4(kb[n][j], kp[n] + r * 64 + (((lane >> 3) ^ ((r >> 1) & 3)) << 4));
    }
#pragma unroll
  for (int n = 0; n < N; ++n) {
    const int r = ((lane >> 4) & 1) * 8 + (lane & 7), sw = (r >> 1) & 3, dsel = (lane >> 3) & 1;
    ldsm_x4_trans(va[n][0], vp[n] + r * 64 + ((dsel ^ sw) << 4));
    ldsm_x4_trans(va[n][1], vp[n] + r * 64 + (((2 + dsel) ^ sw) << 4));
  }
  float sc[N][4];
#pragma unroll
  for (int n = 0; n < N; ++n) {
    const uint32_t a_k0[4] = {aq[n][0][0], 0u, aq[n][0][1], 0u}, a_k1[4] = {aq[n][1][0], 0u, aq[n][1][1], 0u};
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      float c[4] = {0.f, 0.f, 0.f, 0.f}, d[4] = {0.f, 0.f, 0.f, 0.f};
      mma_m16n8k16<bf16>(c, a_k0, kb[n][j][0], kb[n][j][1]);
      mma_m16n8k16<bf16>(d, a_k1, kb[n][j][2], kb[n][j][3]);
      sc[n][2 * j] = c[0] + d[0];
      sc[n][2 * j + 1] = c[1] + d[1];
    }
  }
  // Softmax against a REFERENCE maximum instead of the running one: the reference m is the maximum of the image's first tile and is
  // only raised (with the usual rescale of the state) when some score exceeds it by more than 64 log2-units -- p = 2^(s - m) then
  // stays below 2^64, far inside fp32/bf16 range, and the final o / l is the same quotient.  The common path per tile has no
  // cross-lane maximum (two shuffles), no rescale factor and no state rescale on the dependent chain ldmatrix -> MMA -> ex2 -> MMA; the
  // guard costs one warp vote per image.  Every image decides alone (its own vote), so an image's arithmetic does not depend on the
  // image it shares the warp with (the instantiations stay bitwise equal).
  float mx[N];
#pragma unroll
  for (int n = 0; n < N; ++n) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int key = key0 + (e >> 1) * 8 + 2 * q4 + (e & 1);
      if (padw[n] != nullptr && ((padw[n][key >> 5] >> (key & 31)) & 1u)) sc[n][e] += LOG2E;   // float PAD-key bias +1.0 (Q7), in log2 units
      if (key >= nkeys) sc[n][e] = -INFINITY;                                                  // tail of the last tile
    }
    mx[n] = fmaxf(fmaxf(sc[n][0], sc[n][1]), fmaxf(sc[n][2], sc[n][3]));
  }
#pragma unroll
  for (int n = 0; n < N; ++n) {
    // first tile: m = -inf, and the tile holds a valid key (key0 < nkeys), so some lane sees a finite score and votes
    if (__any_sync(0xffffffffu, mx[n] > st[n].m + margin)) {
      float t = fmaxf(mx[n], __shfl_xor_sync(0xffffffffu, mx[n], 1));
      t = fmaxf(t, __shfl_xor_sync(0xffffffffu, t, 2));          // the quad holds all 16 keys of the tile: the tile maximum, in every lane
      const float m_new = fmaxf(st[n].m, t);
      const float sf = ex2_approx(st[n].m - m_new);              // first tile: 2^-inf = 0 on a zero state
      st[n].m = m_new;
      st[n].ls *= sf;
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int e = 0; e < 4; ++e) st[n].o[mt][e] *= sf;
    }
  }
#pragma unroll
  for (int n = 0; n < N; ++n) {
    float p[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) p[e] = ex2_approx(sc[n][e] - st[n].m);
    st[n].ls += (p[0] + p[1]) + (p[2] + p[3]);
    const uint32_t b0 = pack_bf16x2(p[0], p[1]), b1 = pack_bf16x2(p[2], p[3]);
    mma_m16n8k16<bf16>(st[n].o[0], va[n][0], b0, b1);
    mma_m16n8k16<bf16>(st[n].o[1], va[n][1], b0, b1);
  }
}

// Greedy select of one image by ONE warp, no block barrier: argmax (lowest index on ties, like torch.argmax) and the maximal
// softmax probability 1 / sum exp(l - max) (inference_p.py:77, 84-86 with top_k = 0, top_p = 1: the filter is the identity).
__device__ __forceinline__ void warp_greedy_select(const float* lg, int V, int& token, float& conf) {
  const int lane = threadIdx.x & 31;
  float bv = -INFINITY; int bi = 0x7fffffff;
  for (int i = lane; i < V; i += 32) { const float v = lg[i]; if (v > bv) { bv = v; bi = i; } }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o); const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
  }
  float sum = 0.f;
  for (int i = lane; i < V; i += 32) sum += expf(lg[i] - bv);
  token = bi; conf = 1.0f / warp_sum(sum);
}

// kTrace: developer build of the same kernel that stamps clock64() at phase boundaries (tools/decode_trace.py); the production
// instantiation carries no trace instructions.
// NSTG ring stages; MINB = 2: compact shared-memory layout and a register budget that let two CTAs (of two different clusters,
// i.e. two independent image groups) share an SM, so that one group's dependent phase chain fills the other's stalls.
// kStop: stop at EOS (mdc_decode_state.stop_at_eos).  A template parameter, so that the instantiations without it compile to the code
// they had before the option existed (as a run-time flag its few instructions shifted the register allocation: -1.2 % img/s).
// kPrompt: prompted decoding (mdc_decode_state.prompt_len), a template parameter for the same reason: a prompt step publishes the
// prompt token of column t+1 instead of the selected one and never counts as an EOS.
template <bool kTrace, int NB, int NSTG, int MINB, bool kStop, bool kPrompt>
__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(NT, MINB) decode_fused_kernel(const __grid_constant__ FusedParams P) {
  using Y = Lay<NB, NSTG, NB == 2 || MINB == 2>;
  constexpr int GMX = Y::GMX, NS = Y::NS, STAGE = Y::STAGE;
  // paired K/V hand-overs need ring depth: with four slots the producer can only run one pair ahead and the copies become visible
  // (measured: 10-slot ring 7.95 -> 7.48 ms per launch, 4-slot rings 12.2 -> 13.3 ms)
  constexpr bool KV_PAIRS = NS >= 6;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);      // pointer arithmetic keeps the shared address space
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_rank();
  const int cid = blockIdx.x / CS, n_clusters = gridDim.x / CS;

  __half* xh = (__half*)(smem + Y::OFF_XH); __half* fh = (__half*)(smem + Y::OFF_FH);      // projection operands (fp16)
  float* xres = (float*)(smem + Y::OFF_XRES); float* yrecv = (float*)(smem + Y::OFF_YRECV); float* f2recv = (float*)(smem + Y::OFF_F2RECV);
  float* qs = (float*)(smem + Y::OFF_QS); float* knew = (float*)(smem + Y::OFF_KNEW); float* vnew = (float*)(smem + Y::OFF_VNEW);
  float* ytmp = (float*)(smem + Y::OFF_YTMP); float* ost = (float*)(smem + Y::OFF_OST);
  bf16* qh = (bf16*)(smem + Y::OFF_QH);
  float* lrecv = (float*)(smem + Y::OFF_LRECV); float* selbuf = (float*)(smem + Y::OFF_SEL);
  int* tokbuf = (int*)(smem + Y::OFF_TOK); int* pages = (int*)(smem + Y::OFF_PAGES); uint32_t* padbits = (uint32_t*)(smem + Y::OFF_PADF);
  int* haspad = (int*)(smem + Y::OFF_HASPAD);
  uint32_t* finm = (uint32_t*)(smem + Y::OFF_FIN); volatile int* all_fin = (int*)(smem + Y::OFF_FIN + 8);
  uint32_t* ph_step = (uint32_t*)(smem + Y::OFF_FIN + 12);     // in shared memory: a register live across the group loop costs spills
  int* plen = (int*)(smem + Y::OFF_PLEN);                        // kPrompt only
  const uint32_t bars = sbase + Y::OFF_BARS;
  auto bar = [&](int i) -> uint32_t { return bars + i * 8; };

  if (tid == 0) {
    for (int i = 0; i < NS; ++i) { mbar_init(bar(BAR_FULL + i), 1); mbar_init(bar(BAR_EMPTY + i), 8); }
    for (int i = BAR_O; i < BAR_COUNT; ++i) mbar_init(bar(i), 1);
    *ph_step = 0;
    fence_mbarrier_init();
  }
  // zero the ring and the activation operands once: rows >= G of the operands are multiplied by weights and must be finite
  // (ring bytes that a stage does not fill are only ever stale finite fp16 / bf16 data of earlier stages)
  for (int i = tid; i < (NS * STAGE + 3 * Y::ACT_BYTES) / 16; i += NT) reinterpret_cast<uint4*>(smem + Y::OFF_RING)[i] = make_uint4(0u, 0u, 0u, 0u);
  __syncthreads();
  cluster_sync();

  const float scale = rsqrtf((float)HD) * LOG2E;      // scores in log2 units: p = exp2(s - m)
#ifdef MDC_DEVTOOLS
  const float ref_margin = P.ref_margin;               // tools/ref_margin_check.py: margin 0 = a running maximum, the rescale path on every new maximum
#else
  constexpr float ref_margin = 64.0f;
#endif
  const int L = P.layers, S = P.S;
  const int nck = (S + 15) >> 4;                      // cross-attention key chunks (16 keys each)

  // ring cursors (producer and consumers keep their own copies)
  uint32_t slot = 0, phase = 0;
  uint32_t ph_o = 0, ph_y = 0, ph_f2 = 0, ph_lg = 0, ph_tok = 0;

  for (int grp = cid; grp < P.n_groups; grp += n_clusters) {
    const int img0 = grp * P.G;
    const int G = min(P.G, P.B - img0);
    // ---- per-group init: page ids, PAD flags of the known prefix ---------------------------------------------
    for (int i = tid; i < GMX * 32; i += NT) {
      const int g = i >> 5, j = i & 31;
      pages[i] = (g < G && j < P.pages_per_seq) ? P.page_table[(int64_t)(img0 + g) * P.pages_per_seq + j] : 0;
    }
    for (int i = tid; i < GMX * 8; i += NT) {      // PAD bits of the known prefix (tokens [0, t_begin))
      const int g = i >> 3, w = i & 7;
      uint32_t bits = 0;
      if (g < G)
        for (int b = 0; b < 32 && w * 32 + b < P.t_begin; ++b)
          if (P.tokens[(int64_t)(img0 + g) * P.tokens_ld + w * 32 + b] == P.pad_idx) bits |= 1u << b;
      padbits[i] = bits;
    }
    if (kPrompt)
      for (int i = tid; i < GMX; i += NT) plen[i] = i < G ? P.prompt_len[img0 + i] : 0;
    __syncthreads();
    if (tid < GMX) {
      uint32_t any = 0;
      for (int w = 0; w < 8; ++w) any |= padbits[tid * 8 + w];
      haspad[tid] = any != 0u;
    }
    if (kStop && warp == 0) {      // images with an EOS among the known columns 1..t_begin are finished from the start
      bool f = false;
      if (lane < G)
        for (int c = 1; c <= P.t_begin; ++c) f |= P.tokens[(int64_t)(img0 + lane) * P.tokens_ld + c] == P.eos;
      const uint32_t m = __ballot_sync(0xffffffffu, f);
      if (lane == 0) finm[(P.t_begin + 1) & 1] = m;      // read at step t_begin as "the mask before the previous step"
    }
    __syncthreads();
    cluster_sync();          // no peer may push into this CTA before its buffers are set up for the group

    if (warp == 8) {
      // =================================== PRODUCER WARP ===================================================
      long long prod_wait = 0;
      auto acquire = [&]() -> uint32_t {           // wait until the consumers released the slot
        const long long c0 = kTrace ? clock64() : 0;
        mbar_wait(bar(BAR_EMPTY + slot), phase ^ 1);
        if (kTrace) prod_wait += clock64() - c0;
        return sbase + Y::OFF_RING + slot * STAGE;
      };
      auto advance = [&]() { if (++slot == NS) { slot = 0; phase ^= 1; } };
      // packed weights of (layer l, this CTA): BLOCKS_PER_LAYER consecutive 16 KB blocks in consumption order; a projection of
      // nblk blocks starting at block `first` takes ceil(nblk / NB) stages, each ONE bulk copy of up to NB blocks
      const uint8_t* wl = nullptr;
      auto emit_proj = [&](int first, int nblk) {
        for (int s = 0; s * NB < nblk; ++s) {
          const int here = min(NB, nblk - s * NB);
          const uint32_t st = acquire(); const uint32_t fb = bar(BAR_FULL + slot);
          if (lane == 0) {
            mbar_expect_tx(fb, here * BLK_BYTES);
            bulk_g2s(st, wl + (size_t)(first + s * NB) * BLK_BYTES, here * BLK_BYTES, fb);
          }
          advance();
        }
      };
      // chunk c (16 keys) of the K and V head slices of all images of the group: [image][k|v][16 keys][64 B].  Self-KV: one 2 KB copy
      // per image (its page of the pool).  Cross-K/V is packed in blocks of 8 images ([layer][image / 8][head][chunk][image % 8] x
      // 2 KB), so a group of 8 or 16 images that starts on a multiple of 8 is fetched with one 16 KB copy per block.
      const bool ckv_blocks = (img0 & 7) == 0 && (G & 7) == 0;
      const int nb8 = (P.B + 7) >> 3;
      auto emit_kv = [&](bool cross, int l, int c) {
        const uint32_t st = acquire(); const uint32_t fb = bar(BAR_FULL + slot);
        if (lane == 0) mbar_expect_tx(fb, G * 2048);
        __syncwarp();
        if (cross) {
          const int img = img0 + (ckv_blocks ? lane * 8 : lane);
          const uint8_t* src = P.ckv_pack + (((((size_t)l * nb8 + (img >> 3)) * CS + rank) * nck + c) * 8 + (img & 7)) * 2048;
          if (ckv_blocks) { if (lane < (G >> 3)) bulk_g2s(st + lane * 16384, src, 16384, fb); }
          else if (lane < G) bulk_g2s(st + lane * 2048, src, 2048, fb);
        } else if (lane < G) {
          bulk_g2s(st + lane * 2048, (const uint8_t*)P.kv_pool + (((size_t)pages[lane * 32 + c] * L + l) * CS + rank) * 2048, 2048, fb);
        }
        advance();
      };
      // (deep rings only, KV_PAIRS) Two consecutive chunks as ONE hand-over: both slots' copies complete on the first slot's barrier (the second slot's barrier
      // gets a plain arrival so that its phase keeps step with the ring); the consumers wait once per 32 keys instead of once per 16
      // (a wait on an already complete barrier plus the release and loop cost ~235 of the ~745 cycles a 16-key tile took).
      auto kv_copy = [&](bool cross, int l, int c, uint32_t st, uint32_t fb) {
        if (cross) {
          const int img = img0 + (ckv_blocks ? lane * 8 : lane);
          const uint8_t* src = P.ckv_pack + (((((size_t)l * nb8 + (img >> 3)) * CS + rank) * nck + c) * 8 + (img & 7)) * 2048;
          if (ckv_blocks) { if (lane < (G >> 3)) bulk_g2s(st + lane * 16384, src, 16384, fb); }
          else if (lane < G) bulk_g2s(st + lane * 2048, src, 2048, fb);
        } else if (lane < G) {
          bulk_g2s(st + lane * 2048, (const uint8_t*)P.kv_pool + (((size_t)pages[lane * 32 + c] * L + l) * CS + rank) * 2048, 2048, fb);
        }
      };
      auto emit_kv2 = [&](bool cross, int l, int c) {
        const uint32_t st0 = acquire(); const uint32_t fb0 = bar(BAR_FULL + slot);
        advance();
        const uint32_t st1 = acquire(); const uint32_t fb1 = bar(BAR_FULL + slot);
        advance();
        if (lane == 0) { mbar_expect_tx(fb0, 2 * G * 2048); mbar_arrive(fb1); }
        __syncwarp();
        kv_copy(cross, l, c, st0, fb0);
        kv_copy(cross, l, c + 1, st1, fb0);
      };
      constexpr int PF_AHEAD = 4;                  // chunks of cross-K/V prefetched into L2 ahead of the ring
      auto prefetch_ckv = [&](int l, int c) {
        if (c < nck) {
          const int img = img0 + (ckv_blocks ? lane * 8 : lane);
          const uint8_t* src = P.ckv_pack + (((((size_t)l * nb8 + (img >> 3)) * CS + rank) * nck + c) * 8 + (img & 7)) * 2048;
          if (ckv_blocks) { if (lane < (G >> 3)) bulk_prefetch_l2(src, 16384); }
          else if (lane < G) bulk_prefetch_l2(src, 2048);
        }
      };
      auto emit_kv_all = [&](bool cross, int l, int n) {
        int c = 0;
        if (KV_PAIRS)
          for (; c + 1 < n; c += 2) { emit_kv2(cross, l, c); if (cross) { prefetch_ckv(l, c + PF_AHEAD); prefetch_ckv(l, c + PF_AHEAD + 1); } }
        for (; c < n; ++c) { emit_kv(cross, l, c); if (cross) prefetch_ckv(l, c + PF_AHEAD); }
      };
      for (int t = P.t_begin; t < P.t_end; ++t) {
        // stop at EOS: no stage of step t before the consumers have decided that it runs (from the tokens of step t - 1), so that the
        // ring holds nothing the consumers would not take when the group ends here.  This gives up the producer's lookahead across the
        // step boundary; without stopping the producer never waits here.
        if (kStop) {
          const uint32_t ph = *ph_step;
          mbar_wait(bar(BAR_STEP), ph);
          __syncwarp();
          if (lane == 0) *ph_step = ph ^ 1u;
          if (*all_fin) {
            // the group ends before step t: token columns t+1..t_end and the conf columns of steps t..t_end-1 of the images this CTA
            // selects for become PAD / 0 (never left to what the caller's buffers held).  The producer warp is idle from here on and
            // the consumers wrote only columns <= t; filling here keeps the consumers' register allocation as it was.
            for (int g = (int)rank; g < G; g += CS) {
              int32_t* row = P.tokens + (int64_t)(img0 + g) * P.tokens_ld;
              for (int c = t + 1 + lane; c <= P.t_end; c += 32) row[c] = P.pad_idx;
              if (P.confs)
                for (int c = (t + 3) / 4 + lane; c < (P.t_end + 3) / 4; c += 32) P.confs[(int64_t)(img0 + g) * P.confs_ld + c] = 0.f;
            }
            break;
          }
        }
        const int npg = (t + P.PT - 1) / P.PT;     // pages (= 16-key chunks) holding keys 0..t-1
        for (int l = 0; l < L; ++l) {
          wl = P.wpack + ((size_t)l * CS + rank) * BLOCKS_PER_LAYER * BLK_BYTES;
          emit_proj(0, 3);                                            // in-proj: own head's q rows, k rows, v rows
          for (int c = 0; c < PF_AHEAD; ++c) prefetch_ckv(l, c);      // this layer's first cross-K/V chunks: into L2 during self-attention
          emit_kv_all(false, l, npg);                                 // self-KV pages
          emit_proj(3, 1);                                            // self out-proj rows
          emit_proj(4, 1);                                            // cross-q rows
          emit_kv_all(true, l, nck);                                  // cross K/V chunks
          emit_proj(5, 1);                                            // cross out-proj rows
          emit_proj(6, 8);                                            // FFN1: own hidden rows
          emit_proj(14, 8);                                           // FFN2: K-split over the own hidden columns
        }
        // vocabulary head rows: [0,32) of the own 40 as one block, [32,40) as an 8-row block (same stage with NB = 2, the next otherwise)
        {
          const uint8_t* hp = P.wpack + (size_t)L * CS * BLOCKS_PER_LAYER * BLK_BYTES + (size_t)rank * HEAD_PACK_BYTES;
          uint32_t st = acquire(); uint32_t fb = bar(BAR_FULL + slot);
          if (NB == 2) {
            if (lane == 0) { mbar_expect_tx(fb, HEAD_PACK_BYTES); bulk_g2s(st, hp, HEAD_PACK_BYTES, fb); }
          } else {
            if (lane == 0) { mbar_expect_tx(fb, BLK_BYTES); bulk_g2s(st, hp, BLK_BYTES, fb); }
            advance(); st = acquire(); fb = bar(BAR_FULL + slot);
            if (lane == 0) { mbar_expect_tx(fb, 8 * 512); bulk_g2s(st, hp + BLK_BYTES, 8 * 512, fb); }
          }
          advance();
        }
      }
      if (kTrace && lane == 0 && blockIdx.x == 0) P.trace[202] = prod_wait;
    } else {
      // =================================== CONSUMER WARPS ==================================================
      long long cons_wait = 0, exch_wait = 0;
      int wait_phase = 0;                       // trace build: which phase the stage waits of warp 0 are charged to (trace[210 + phase])
      auto stage_wait = [&]() -> uint32_t {
        const long long c0 = kTrace ? clock64() : 0;
        mbar_wait(bar(BAR_FULL + slot), phase);
        if (kTrace) { const long long d = clock64() - c0; cons_wait += d; if (tid == 0 && blockIdx.x == 0) P.trace[210 + wait_phase] += d; }
        return sbase + Y::OFF_RING + slot * STAGE;
      };
      auto xwait = [&](int which, uint32_t& ph) {    // wait for a push-style exchange
        const long long c0 = kTrace ? clock64() : 0;
        mbar_wait(bar(which), ph); ph ^= 1;
        if (kTrace) exch_wait += clock64() - c0;
      };
      // A stage is released by the warps that read it: the empty barrier counts 8 arrivals, a stage with k user warps gets
      // 8/k from each of them (`weight`); the other warps neither wait for the stage nor arrive, they only advance the cursor.
      auto stage_release = [&](uint32_t weight = 1) {
        __syncwarp();
        if (lane == 0) mbar_arrive_n(bar(BAR_EMPTY + slot), weight);
        if (++slot == NS) { slot = 0; phase ^= 1; }
      };
      auto stage_skip = [&]() { if (++slot == NS) { slot = 0; phase ^= 1; } };
      const int fg = lane >> 2, fq = lane & 3;       // MMA fragment coordinates: row group, image pair
      int trace_n = 0;
      auto TRACE = [&](int t_now) { if (kTrace && tid == 0 && blockIdx.x == 0 && t_now == P.trace_t) P.trace[trace_n++] = clock64(); };
      auto FINE = [&](int l_now, int t_now, int idx) {   // trace build: fine stamps of layer 2 into trace[100 + idx] by lane 0 of the calling warp
        if (kTrace && lane == 0 && blockIdx.x == 0 && t_now == P.trace_t && l_now == 2) P.trace[100 + idx] = clock64();
      };
      const int gi_t = tid >> 5, c_t = tid & 31;     // (image [+ 8], channel) coordinates of the elementwise phases
      constexpr int APP0 = NCT - GMX * 8;           // first thread of the KV-append crew (the last GMX * 8 consumer threads)
      // A projection of nblk 32-row weight blocks, NB blocks per stage: block b belongs to warp pair b % 4 (16 rows per warp).
      // body(b, block address, m-tile 0 / 1) runs in the two warps of the pair; every other warp only advances its ring cursor.
      auto proj_blocks = [&](int nblk, auto&& body) {
        const int pr = warp >> 1;
        for (int s = 0; s * NB < nblk; ++s) {
          const int j = (pr - s * NB) & 3, b = s * NB + j;
          if (j < NB && b < nblk) {
            const uint32_t users = 2u * (uint32_t)min(NB, nblk - s * NB);
            const uint32_t st = stage_wait();
            body(b, st + j * BLK_BYTES, warp & 1);
            stage_release(8u / users);
          } else stage_skip();
        }
      };
      // push this CTA's [G][32] slice in ytmp into every peer's yrecv columns [32*rank, +32)
      auto push_y = [&](int img, float v) {
        if (img < G) {
          const uint32_t off = sbase + Y::OFF_YRECV + (img * DM + 32 * rank + c_t) * 4;
#pragma unroll
          for (int p = 0; p < CS; ++p) st_async_b32(mapa(off, p), __float_as_uint(v), mapa(bar(BAR_Y), p));
        }
      };
      auto wait_y = [&]() {
        if (tid == 0) mbar_expect_tx(bar(BAR_Y), G * DM * 4);
        xwait(BAR_Y, ph_y);
      };
      // x = LN(xres + yrecv): warp w owns images w (and w + 8); writes xres and the fp16 operand
      auto layer_norm = [&](const float* lnw, const float* lnb, bool fence_appends = false, int l_now = -1, int t_now = -1, int fi = 0) {
        if (warp == 0) FINE(l_now, t_now, fi);
        // this layer's KV append: the generic->async proxy fence (~1200 cycles) of the appending threads overlaps the exchange latency
        if (fence_appends && tid >= APP0 && tid - APP0 < G * 8) fence_proxy_async();
        float gw[8], gb[8];
        if (warp < G) {
#pragma unroll
          for (int j = 0; j < 8; ++j) { gw[j] = __ldg(lnw + lane + 32 * j); gb[j] = __ldg(lnb + lane + 32 * j); }
        }
        wait_y();
        if (warp == 0) FINE(l_now, t_now, fi + 1);
        // the warp's two images in lockstep: each image keeps its own operation sequence (results unchanged), but the two shuffle
        // butterflies and the two reciprocal square roots overlap instead of running one after the other (900 cycles per image)
        float v[NB][8], sm[NB], mean[NB], rstd[NB];
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) {
          const int img = min(warp + 8 * nb, GMX - 1);
          sm[nb] = 0.f;
#pragma unroll
          for (int j = 0; j < 8; ++j) { v[nb][j] = xres[img * DM + lane + 32 * j] + yrecv[img * DM + lane + 32 * j]; sm[nb] += v[nb][j]; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
          for (int nb = 0; nb < NB; ++nb) sm[nb] += __shfl_xor_sync(0xffffffffu, sm[nb], o);
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) {
          mean[nb] = sm[nb] * (1.0f / DM);
          float q = 0.f;
#pragma unroll
          for (int j = 0; j < 8; ++j) { const float d = v[nb][j] - mean[nb]; q += d * d; }
          sm[nb] = q;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
          for (int nb = 0; nb < NB; ++nb) sm[nb] += __shfl_xor_sync(0xffffffffu, sm[nb], o);
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) rstd[nb] = 1.0f / sqrtf(sm[nb] * (1.0f / DM) + 1e-5f);
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) {
          const int img = warp + 8 * nb;
          if (img < G) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int c = lane + 32 * j;
              const float xn = (v[nb][j] - mean[nb]) * rstd[nb] * gw[j] + gb[j];
              xres[img * DM + c] = xn;
              xh[img * XP + c] = f16_sat(xn);
            }
          }
        }
        if (warp == 0) FINE(l_now, t_now, fi + 2);
        cbar();
        if (warp == 0) FINE(l_now, t_now, fi + 3);
      };
      // attention output of image `img` (lane = channel) -> fp16 pairs into every peer's oh columns [32*rank, +32); lane j < 16
      // sends channels 2j, 2j+1 to peers 0..3, lane 16 + j the same pair to peers 4..7
      auto push_o = [&](int img, float o) {
        const int j = lane & 15;
        const float v0 = __shfl_sync(0xffffffffu, o, 2 * j), v1 = __shfl_sync(0xffffffffu, o, 2 * j + 1);
        if (img < G) {
          const uint32_t val = pack_f16x2_sat(v0, v1);
          const uint32_t off = sbase + Y::OFF_OH + (img * XP + 32 * rank + 2 * j) * 2;
          const int p0 = (lane >> 4) * 4;
#pragma unroll
          for (int p = 0; p < 4; ++p) st_async_b32(mapa(off, p0 + p), val, mapa(bar(BAR_O), p0 + p));
        }
      };
      auto wait_o = [&]() {
        if (tid == 0) mbar_expect_tx(bar(BAR_O), G * DM * 2);
        xwait(BAR_O, ph_o);
      };
      // a 32-row projection of the gathered operand bh -> ytmp (+bias) -> pushed to all peers
      auto proj32_push = [&](uint32_t bh, const float* bias) {
        float b0 = 0.f, b1 = 0.f;
        if (warp < 2) { b0 = __ldg(bias + rank * 32 + warp * 16 + fg); b1 = __ldg(bias + rank * 32 + warp * 16 + fg + 8); }
        proj_blocks(1, [&](int, uint32_t blk, int mt) {
          float acc[NB][4];
          mma_mtile<32, NB>(blk, mt * 16, bh, acc);
          const int f = mt * 16 + fg;
#pragma unroll
          for (int nb = 0; nb < NB; ++nb) {
            float* y = ytmp + (8 * nb + 2 * fq) * 32 + f;
            y[0] = acc[nb][0] + b0; y[32] = acc[nb][1] + b0; y[8] = acc[nb][2] + b1; y[40] = acc[nb][3] + b1;
          }
        });
        cbar();
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) push_y(gi_t + 8 * nb, ytmp[(gi_t + 8 * nb) * 32 + c_t]);
      };
      // Attention of head `rank` for the images of this warp (image `warp`, and `warp + 8` with NB = 2) over nchunk 16-key chunks:
      // the warp keeps the running softmax state of its images in registers across the chunks (every warp reads every chunk stage:
      // its own images' panels), then stages the un-normalised output, running maximum and denominator in `ost` (fragment order ->
      // channel order).  One image = one warp = one fixed operation sequence: results do not depend on the batch or the variant.
      auto attention = [&](int nchunk, int nkeys, bool use_pad, int l_now, int t_now) {
        AttnState as[NB];
        uint32_t aq[NB][2][2];
        const uint32_t* padw[NB];
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) {
          const int img = warp + 8 * nb;
          as[nb].m = -INFINITY; as[nb].ls = 0.f;
#pragma unroll
          for (int mt = 0; mt < 2; ++mt)
#pragma unroll
            for (int e = 0; e < 4; ++e) as[nb].o[mt][e] = 0.f;
          padw[nb] = (use_pad && img < G && haspad[img]) ? padbits + img * 8 : nullptr;
          if (img < G) build_q_frag(qh + img * 32, aq[nb]);
          else { aq[nb][0][0] = aq[nb][0][1] = aq[nb][1][0] = aq[nb][1][1] = 0u; }
        }
        const bool two = NB == 2 && warp + 8 < G;
        // (probing the next stage's barrier early, so that its ~150-cycle try_wait overlaps the current chunk's MMA chain, was
        //  measured SLOWER: 12.73 -> 13.26 ms per launch, profiles/r2 notes)
        auto tile = [&](uint32_t st, int c) {          // one 16-key tile of the warp's images from the stage at `st`
          if (warp < G) {
            bool done = false;
            if constexpr (NB == 2) {
              if (two) {
                const uint32_t kp[2] = {st + warp * 2048u, st + (warp + 8) * 2048u};
                const uint32_t vp[2] = {kp[0] + 1024u, kp[1] + 1024u};
                attn_tile<2>(kp, vp, aq, c * 16, nkeys, padw, as, ref_margin);
                done = true;
              }
            }
            if (!done) {
              const uint32_t kp[1] = {st + warp * 2048u}, vp[1] = {kp[0] + 1024u};
              const uint32_t aq1[1][2][2] = {{{aq[0][0][0], aq[0][0][1]}, {aq[0][1][0], aq[0][1][1]}}};
              const uint32_t* pw1[1] = {padw[0]};
              AttnState a1[1] = {as[0]};
              attn_tile<1>(kp, vp, aq1, c * 16, nkeys, pw1, a1, ref_margin);
              as[0] = a1[0];
            }
          }
        };
        int c = 0;
        if (KV_PAIRS)
        for (; c + 1 < nchunk; c += 2) {               // two chunks per hand-over: one wait (the first slot's barrier covers both copies)
          if (warp == 0 && c < 16) FINE(l_now, t_now, 20 + (c >> 1) * 3);
          const uint32_t st0 = stage_wait();
          const uint32_t st1 = sbase + Y::OFF_RING + (slot + 1 == NS ? 0u : slot + 1) * STAGE;
          if (warp == 0 && c < 16) FINE(l_now, t_now, 21 + (c >> 1) * 3);
          tile(st0, c);
          tile(st1, c + 1);
          stage_release();
          stage_release();
          if (warp == 0 && c < 16) FINE(l_now, t_now, 22 + (c >> 1) * 3);
        }
        for (; c < nchunk; ++c) {
          const uint32_t st = stage_wait();
          tile(st, c);
          stage_release();
        }
#pragma unroll
        for (int nb = 0; nb < NB; ++nb) {
          const int img = warp + 8 * nb;
          if (img < G) {
            float lt = as[nb].ls;
            lt += __shfl_xor_sync(0xffffffffu, lt, 1);
            lt += __shfl_xor_sync(0xffffffffu, lt, 2);
            float* ob = ost + img * OSTR;
            if (fq == 0) { ob[fg] = as[nb].o[0][0]; ob[fg + 8] = as[nb].o[0][2]; ob[fg + 16] = as[nb].o[1][0]; ob[fg + 24] = as[nb].o[1][2]; }
            if (lane == 0) { ob[32] = as[nb].m; ob[33] = lt; }
          }
        }
        __syncwarp();
      };

      for (int t = P.t_begin; t < P.t_end; ++t) {
        const int npg = (t + P.PT - 1) / P.PT;
        // ---- stop at EOS: finished mask before step t (bit g: image g has emitted EOS, or had one among columns 1..t_begin) and the
        //      decision whether step t runs.  Every CTA of the cluster received the same tokens, so every CTA decides the same. -------
        if (kStop && warp == 0) {
          const bool eos_now = t > P.t_begin && lane < G && tokbuf[(t & 1) * GMX + lane] == P.eos && !(kPrompt && t <= plen[lane]);
          const uint32_t f = finm[(t + 1) & 1] | __ballot_sync(0xffffffffu, eos_now);
          if (lane == 0) {
            finm[t & 1] = f;
            *all_fin = f == (1u << G) - 1u;
            mbar_arrive(bar(BAR_STEP));
          }
        }
        // ---- embedding + positional row (model.py:98-101); PAD flag of the token at position t --------------
        if (warp < G) {
          float pz[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) pz[j] = __ldg(P.pos + (int64_t)t * DM + lane + 32 * j);
#pragma unroll
          for (int nb = 0; nb < NB; ++nb) {
            const int img = warp + 8 * nb;
            if (img < G) {
              const int tok = (P.forced || t == P.t_begin) ? __ldcg(P.tokens + (int64_t)(img0 + img) * P.tokens_ld + t) : tokbuf[(t & 1) * GMX + img];
              if (lane == 0 && tok == P.pad_idx) { padbits[img * 8 + (t >> 5)] |= 1u << (t & 31); haspad[img] = 1; }
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const int c = lane + 32 * j;
                const float x = __ldg(P.emb + (int64_t)tok * DM + c) + pz[j];
                xres[img * DM + c] = x;
                xh[img * XP + c] = f16_sat(x);
              }
            }
          }
        }
        cbar();
        if (kStop && *all_fin) break;
        for (int l = 0; l < L; ++l) {
          TRACE(t);   // 0: layer start
          if (kTrace) wait_phase = 0;
          // ---- self-attention in-proj: own head's q (warps 0-1), k (warps 2-3), v (warps 4-5), one 32-row block each ------
          {
            const float* bi = P.b_in[l];
            const int part = warp >> 1;                  // 0 q, 1 k, 2 v (3: no projection work)
            float b0 = 0.f, b1 = 0.f;
            if (part < 3) { const int r0 = part * DM + rank * HD + (warp & 1) * 16 + fg; b0 = __ldg(bi + r0); b1 = __ldg(bi + r0 + 8); }
            proj_blocks(3, [&](int pt, uint32_t blk, int mt) {
              float acc[NB][4];
              mma_mtile<32, NB>(blk, mt * 16, sbase + Y::OFF_XH, acc);
              const int f = mt * 16 + fg;
#pragma unroll
              for (int nb = 0; nb < NB; ++nb) {
                const int o = (8 * nb + 2 * fq) * 32 + f;
                if (pt == 0) {       // q, pre-scaled
                  const float q0 = (acc[nb][0] + b0) * scale, q1 = (acc[nb][1] + b0) * scale, q2 = (acc[nb][2] + b1) * scale, q3 = (acc[nb][3] + b1) * scale;
                  const bf16 r0 = __float2bfloat16_rn(q0), r1 = __float2bfloat16_rn(q1), r2 = __float2bfloat16_rn(q2), r3 = __float2bfloat16_rn(q3);
                  qh[o] = r0; qh[o + 32] = r1; qh[o + 8] = r2; qh[o + 40] = r3;
                  // the step's own key meets the same bf16 query as the cached keys
                  qs[o] = __bfloat162float(r0); qs[o + 32] = __bfloat162float(r1); qs[o + 8] = __bfloat162float(r2); qs[o + 40] = __bfloat162float(r3);
                } else {             // k / v, rounded to the cache precision
                  float* dst = pt == 1 ? knew : vnew;
                  dst[o] = __bfloat162float(__float2bfloat16_rn(acc[nb][0] + b0));
                  dst[o + 32] = __bfloat162float(__float2bfloat16_rn(acc[nb][1] + b0));
                  dst[o + 8] = __bfloat162float(__float2bfloat16_rn(acc[nb][2] + b1));
                  dst[o + 40] = __bfloat162float(__float2bfloat16_rn(acc[nb][3] + b1));
                }
              }
            });
          }
          cbar();
          TRACE(t);   // 1: in-proj done
          // append k_t, v_t (bf16) to the paged cache: 16-byte stores, 4 per (image, k|v), by the last warps.  The proxy fence that
          // orders them before the TMA reads of the page (one step later) costs ~1200 cycles; the same threads issue it while they
          // wait for the out-projection exchange (layer_norm), where its latency hides behind the exchange's.
          if (tid >= APP0 && tid - APP0 < G * 8) {
            const int at = tid - APP0;
            const int g = at >> 3, which = (at >> 2) & 1, ch = at & 3;
            const float* src = (which ? vnew : knew) + g * 32 + ch * 8;
            const float4 a = *reinterpret_cast<const float4*>(src), b = *reinterpret_cast<const float4*>(src + 4);
            uint4 o; o.x = pack_bf16x2(a.x, a.y); o.y = pack_bf16x2(a.z, a.w); o.z = pack_bf16x2(b.x, b.y); o.w = pack_bf16x2(b.z, b.w);
            const int page = pages[g * 32 + t / P.PT];
            const int r = t % P.PT;      // pool: [page][layer][head][k|v][16 tokens][32]; chunk ch of token r at ch ^ ((r >> 1) & 3) (common.cuh kv_chunk)
            bf16* dst = P.kv_pool + ((((int64_t)page * L + l) * CS + rank) * 2 + which) * (int64_t)(P.PT * HD) + r * HD + ((ch ^ ((r >> 1) & 3)) << 3);
            *reinterpret_cast<uint4*>(dst) = o;
          }
          TRACE(t);   // 2: append
          // ---- self-attention, head `rank`: keys [0,t) from the paged cache in chunks of one page, then the step's own key (still in
          //      shared memory) joins as one more online-softmax term ---------------------------------------------------------------
          if (kTrace) wait_phase = 1;
          attention(npg, t, true, -1, t);
          TRACE(t);   // 3: self attention
#pragma unroll
          for (int nb = 0; nb < NB; ++nb) {
            const int img = warp + 8 * nb;
            float out = 0.f;
            if (img < G) {
              float s_own = warp_sum(qs[img * 32 + lane] * knew[img * 32 + lane]);
              if ((padbits[img * 8 + (t >> 5)] >> (t & 31)) & 1u) s_own += LOG2E;
              const float v_own = vnew[img * 32 + lane];
              if (npg == 0) out = v_own;                     // t = 0: the own key is the only key
              else {
                const float* ob = ost + img * OSTR;
                const float m_run = ob[32], l_run = ob[33];
                const float mf = fmaxf(m_run, s_own);
                const float wr = exp2f(m_run - mf), wo = exp2f(s_own - mf);
                out = fmaf(ob[lane], wr, v_own * wo) / fmaf(l_run, wr, wo);
              }
            }
            push_o(img, out);
          }
          // this layer's KV append: the generic->async proxy fence (~1200 cycles) of the appending threads runs while they wait for the
          // attention-output gather (it used to sit at the head of LayerNorm 1, which was ~1000 cycles longer than LayerNorm 2)
          if (tid >= APP0 && tid - APP0 < G * 8) fence_proxy_async();
          wait_o();
          TRACE(t);   // 4: o gathered
          // ---- self out-proj slice -> all-gather -> LN1 ------------------------------------------------------------
          if (kTrace) wait_phase = 2;
          proj32_push(sbase + Y::OFF_OH, P.b_so[l]);
          TRACE(t);   // 5: out-proj pushed
          layer_norm(P.ln1w[l], P.ln1b[l]);
          TRACE(t);   // 6: LN1

          if (kTrace) wait_phase = 3;
          // ---- cross-attention query slice -------------------------------------------------------------------------
          {
            const float* bc = P.b_ca[l];
            float b0 = 0.f, b1 = 0.f;
            if (warp < 2) { b0 = __ldg(bc + rank * 32 + warp * 16 + fg); b1 = __ldg(bc + rank * 32 + warp * 16 + fg + 8); }
            proj_blocks(1, [&](int, uint32_t blk, int mt) {
              float acc[NB][4];
              mma_mtile<32, NB>(blk, mt * 16, sbase + Y::OFF_XH, acc);
              const int f = mt * 16 + fg;
#pragma unroll
              for (int nb = 0; nb < NB; ++nb) {
                bf16* q = qh + (8 * nb + 2 * fq) * 32 + f;
                q[0] = __float2bfloat16_rn((acc[nb][0] + b0) * scale); q[32] = __float2bfloat16_rn((acc[nb][1] + b0) * scale);
                q[8] = __float2bfloat16_rn((acc[nb][2] + b1) * scale); q[40] = __float2bfloat16_rn((acc[nb][3] + b1) * scale);
              }
            });
          }
          cbar();
          TRACE(t);   // 7: cross q
          // ---- cross-attention over the S memory keys (HBM/L2-resident cross-K/V), 16-key chunks ------------------------------
          if (kTrace) wait_phase = 4;
          attention(nck, S, false, l, t);
          TRACE(t);   // 8: cross attention
#pragma unroll
          for (int nb = 0; nb < NB; ++nb) {
            const int img = warp + 8 * nb;
            float out = 0.f;
            if (img < G) { const float* ob = ost + img * OSTR; out = ob[lane] / ob[33]; }
            push_o(img, out);
          }
          wait_o();
          TRACE(t);   // 9: o gathered
          if (kTrace) wait_phase = 5;
          proj32_push(sbase + Y::OFF_OH, P.b_co[l]);
          TRACE(t);   // 10: cross out-proj pushed
          layer_norm(P.ln2w[l], P.ln2b[l], false, l, t, 60);
          TRACE(t);   // 11: LN2

          if (kTrace) wait_phase = 6;
          // ---- FFN1: own 256 hidden units as 8 blocks of 32 rows (block b -> warp pair b % 4), ReLU, kept local as the FFN2 operand ----
          {
            const float* bf = P.b_f1[l] + rank * FS + (warp & 1) * 16 + fg;
            const int pr = warp >> 1;
            const float ba0 = __ldg(bf + pr * 32), ba1 = __ldg(bf + pr * 32 + 8), bb0 = __ldg(bf + (pr + 4) * 32), bb1 = __ldg(bf + (pr + 4) * 32 + 8);
            proj_blocks(8, [&](int b, uint32_t blk, int mt) {
              const float b0 = b < 4 ? ba0 : bb0, b1 = b < 4 ? ba1 : bb1;
              float acc[NB][4];
              mma_mtile<32, NB>(blk, mt * 16, sbase + Y::OFF_XH, acc);
              const int h = b * 32 + mt * 16 + fg;
#pragma unroll
              for (int nb = 0; nb < NB; ++nb) {
                const int r = 8 * nb + 2 * fq;
                fh[r * XP + h] = f16_sat(fmaxf(acc[nb][0] + b0, 0.f)); fh[(r + 1) * XP + h] = f16_sat(fmaxf(acc[nb][1] + b0, 0.f));
                fh[r * XP + h + 8] = f16_sat(fmaxf(acc[nb][2] + b1, 0.f)); fh[(r + 1) * XP + h + 8] = f16_sat(fmaxf(acc[nb][3] + b1, 0.f));
              }
            });
          }
          cbar();
          TRACE(t);   // 12: FFN1
          if (kTrace) wait_phase = 7;
          // ---- FFN2 as a K-split, 32 output features per block: partial sums pushed straight to the CTA that owns the columns ----
          proj_blocks(8, [&](int b, uint32_t blk, int mt) {
            float acc[NB][4];
            mma_mtile<32, NB>(blk, mt * 16, sbase + Y::OFF_FH, acc);
            const int f = mt * 16 + fg;                                // feature within the block of acc[.][0..1]; +8 for acc[.][2..3]
            const uint32_t peer = (uint32_t)b;                         // block b = the 32-column slice of CTA b
            const uint32_t rb = mapa(bar(BAR_F2), peer);
            const uint32_t base = mapa(sbase + Y::OFF_F2RECV + (rank * GMX * 32 + f) * 4, peer);
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) {
              const int i0 = 8 * nb + 2 * fq;
              if (i0 < G) { st_async_b32(base + i0 * 128, __float_as_uint(acc[nb][0]), rb); st_async_b32(base + i0 * 128 + 32, __float_as_uint(acc[nb][2]), rb); }
              if (i0 + 1 < G) { st_async_b32(base + (i0 + 1) * 128, __float_as_uint(acc[nb][1]), rb); st_async_b32(base + (i0 + 1) * 128 + 32, __float_as_uint(acc[nb][3]), rb); }
            }
          });
          TRACE(t);   // 13: FFN2 issued
          {  // reduce the 8 partial slices of the own 32 columns, add bias, all-gather, LN3
            const float b2 = __ldg(P.b_f2[l] + rank * 32 + c_t);
            if (tid == 0) mbar_expect_tx(bar(BAR_F2), G * DM * 4);
            xwait(BAR_F2, ph_f2);
#pragma unroll
            for (int nb = 0; nb < NB; ++nb) {
              const int img = gi_t + 8 * nb;
              float a = b2;
              if (img < G) {
#pragma unroll
                for (int p = 0; p < CS; ++p) a += f2recv[(p * GMX + img) * 32 + c_t];
              }
              push_y(img, a);
            }
          }
          TRACE(t);   // 14: FFN2 reduced + pushed
          layer_norm(P.ln3w[l], P.ln3b[l], false, l, t, 64);
          TRACE(t);   // 15: LN3

        }
          if (kTrace) wait_phase = 8;
        // ---- vocabulary head: own 40 rows -> logits to the caller's tensor and to the CTA that selects for the image ---
        const bool want_conf = P.confs && (t % 4 == 0);
        const bool need_select = !P.forced || want_conf;
        {
          const int r0 = rank * VSL;
          float b0 = 0.f, b1 = 0.f;
          const int row_a = warp * 16 + fg, row_b = row_a + 8;
          const bool va = warp < 3 && row_a < VSL && r0 + row_a < P.vocab, vb = warp < 3 && row_b < VSL && r0 + row_b < P.vocab;
          if (va) b0 = __ldg(P.b_out + r0 + row_a);
          if (vb) b1 = __ldg(P.b_out + r0 + row_b);
          // rows [0,32) of the own 40 are one block (warps 0-1), rows [32,40) an 8-row block (warp 2: the upper half of its 16-row
          // MMA tile reads the neighbouring k-block -- finite weights feeding accumulator rows that are never used)
          auto head_out = [&](float (&acc)[NB][4]) {
#pragma unroll
            for (int nb = 0; nb < NB; ++nb)
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int img = 8 * nb + 2 * fq + (e & 1); const bool hi8 = e >= 2;
                const bool valid = (hi8 ? vb : va) && img < G;
                if (valid) {
                  const int row = hi8 ? row_b : row_a;
                  const float lg = acc[nb][e] + (hi8 ? b1 : b0);
                  if (P.logits_out) P.logits_out[(int64_t)(img0 + img) * P.logits_img_stride + (int64_t)(t + P.logits_row_offset) * P.vocab + r0 + row] = lg;
                  // the CTA that selects for image img is img % 8; it keeps one [CS][VSL] receive block per owned image
                  if (need_select) st_async_b32(mapa(sbase + Y::OFF_LRECV + ((nb * CS + rank) * VSL + row) * 4, img & 7), __float_as_uint(lg), mapa(bar(BAR_LG), img & 7));
                }
              }
          };
          if (NB == 2) {            // both blocks in one stage: users warps 0, 1 (weight 3 each) and 2 (weight 2)
            if (warp < 3) {
              const uint32_t st = stage_wait();
              float acc[NB][4];
              if (warp < 2) mma_mtile<32, NB>(st, warp * 16, sbase + Y::OFF_XH, acc);
              else mma_mtile<8, NB>(st + BLK_BYTES, 0, sbase + Y::OFF_XH, acc);
              head_out(acc);
              stage_release(warp < 2 ? 3 : 2);
            } else stage_skip();
          } else {
            if (warp < 2) {
              const uint32_t st = stage_wait();
              float acc[NB][4];
              mma_mtile<32, NB>(st, warp * 16, sbase + Y::OFF_XH, acc);
              head_out(acc);
              stage_release(4);
            } else stage_skip();
            if (warp == 2) {
              const uint32_t st = stage_wait();
              float acc[NB][4];
              mma_mtile<8, NB>(st, 0, sbase + Y::OFF_XH, acc);
              head_out(acc);
              stage_release(8);
            } else stage_skip();
          }
        }
        cbar();       // the next step's embedding overwrites the operand rows the head MMAs of warps 0-2 are reading (in teacher-forced
                      // mode nothing else orders the two: no select, no token exchange)
        TRACE(t);     // head done
        // ---- select: CTA `rank` owns images `rank` (and `rank + 8`) ---------------------------------------------------
        if (need_select && (int)rank < G) {
          const int V = P.vocab;
          const int n_own = ((int)rank + 8 < G && NB > 1) ? 2 : 1;
          if (tid == 0) mbar_expect_tx(bar(BAR_LG), n_own * V * 4);
          mbar_wait(bar(BAR_LG), ph_lg);
          ph_lg ^= 1;
          auto publish = [&](int img, int token, float conf) {     // one thread: token to the caller's buffer and to every peer
            if (kStop && ((finm[t & 1] >> img) & 1u)) { token = P.pad_idx; conf = 0.f; }    // finished before step t
            const bool prompt_step = kPrompt && t + 1 <= plen[img];     // column t+1 holds the prompt: exchange it, leave it alone
            if (prompt_step) token = __ldcg(P.tokens + (int64_t)(img0 + img) * P.tokens_ld + t + 1);
            if (!P.forced) {
              if (!prompt_step) P.tokens[(int64_t)(img0 + img) * P.tokens_ld + t + 1] = token;
              const uint32_t off = sbase + Y::OFF_TOK + ((((t + 1) & 1) * GMX) + img) * 4;
#pragma unroll
              for (int p = 0; p < CS; ++p) st_async_b32(mapa(off, p), (uint32_t)token, mapa(bar(BAR_TOK), p));
            }
            if (want_conf) P.confs[(int64_t)(img0 + img) * P.confs_ld + t / 4] = conf;
          };
          if (P.top_k == 0 && P.top_p == 1.0f) {
            // greedy: one warp per owned image straight from the receive buffer ([src][VSL] is vocabulary order), no block barrier
            if (warp < n_own) {
              int token; float conf;
              warp_greedy_select(lrecv + warp * CS * VSL, V, token, conf);
              if (lane == 0) publish(rank + 8 * warp, token, conf);
            }
          } else {
            int Vp2 = 1; while (Vp2 < V) Vp2 <<= 1;
            float* lg = selbuf; float* srt = selbuf + CS * VSL;
            const bool sample = P.uniforms != nullptr;
            for (int nb = 0; nb < n_own; ++nb) {
              const int img = rank + 8 * nb;
              for (int i = tid; i < V; i += NCT) lg[i] = lrecv[nb * CS * VSL + i];
              cbar();
              const float u = sample ? P.uniforms[(int64_t)(img0 + img) * P.uniforms_ld + t] : 0.f;
              int token; float conf;
              select_from_logits(lg, srt, V, Vp2, P.top_k, P.top_p, sample, u, token, conf);
              if (tid == 0) publish(img, token, conf);
              if (nb + 1 < n_own) cbar();      // the scratch is reused by the second image
            }
          }
        }
        if (!P.forced) {
          if (tid == 0) mbar_expect_tx(bar(BAR_TOK), G * 4);
          xwait(BAR_TOK, ph_tok);
        }
        TRACE(t);     // tokens exchanged
      }
      if (kTrace && tid == 0 && blockIdx.x == 0) { P.trace[200] = cons_wait; P.trace[201] = exch_wait; }
    }
  }
  // no CTA may exit while a peer can still push into its shared memory
  __syncthreads();
  cluster_sync();
}

// ---- pack kernels: global-memory images of what the kernel wants in shared memory -----------------------------------
// Weight block (R rows x 256 k, fp16): [4 k-blocks][R rows][128 B], the 16-byte chunk c of row i stored at chunk c ^ (i & 7)
// (the layout a SWIZZLE_128B tensor-map load would produce, which mma_mtile's ldmatrix addressing expects).
struct PackArgs {
  const __half* w[8][6];     // per layer: self in-proj [3*DM][DM], self out [DM][DM], cross in-proj [3*DM][DM] (rows [0,DM) = q), cross out, FFN1 [FFN][DM], FFN2 [DM][FFN]
  const __half* head;        // [vocab][DM]
  int layers, vocab;
};

__global__ void pack_weights_kernel(PackArgs a, uint4* __restrict__ out, size_t n_chunks) {
  const size_t layer_bytes = (size_t)a.layers * CS * BLOCKS_PER_LAYER * BLK_BYTES;
  for (size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x; id < n_chunks; id += (size_t)gridDim.x * blockDim.x) {
    const size_t off = id * 16;
    const __half* src = nullptr;
    if (off < layer_bytes) {
      const int blk = (int)(off / BLK_BYTES), within = (int)(off % BLK_BYTES);
      const int l = blk / (CS * BLOCKS_PER_LAYER), r = (blk / BLOCKS_PER_LAYER) % CS, b = blk % BLOCKS_PER_LAYER;
      const int kb = within / 4096, i = (within % 4096) / 128, pc = (within % 128) / 16;
      const int k0 = kb * 64 + ((pc ^ (i & 7)) << 3);
      if (b < 3) src = a.w[l][0] + (size_t)(b * DM + r * HD + i) * DM + k0;
      else if (b == 3) src = a.w[l][1] + (size_t)(r * 32 + i) * DM + k0;
      else if (b == 4) src = a.w[l][2] + (size_t)(r * 32 + i) * DM + k0;
      else if (b == 5) src = a.w[l][3] + (size_t)(r * 32 + i) * DM + k0;
      else if (b < 14) src = a.w[l][4] + (size_t)(r * FS + (b - 6) * 32 + i) * DM + k0;
      else src = a.w[l][5] + (size_t)((b - 14) * 32 + i) * FFN + r * FS + k0;
    } else {
      const size_t hoff = off - layer_bytes;
      const int r = (int)(hoff / HEAD_PACK_BYTES), within = (int)(hoff % HEAD_PACK_BYTES);
      int kb, i, row;
      if (within < BLK_BYTES) { kb = within / 4096; i = (within % 4096) / 128; row = r * VSL + i; }
      else { const int w2 = within - BLK_BYTES; kb = w2 / 1024; i = (w2 % 1024) / 128; row = r * VSL + 32 + i; }
      const int pc = (within % 128) / 16;
      const int k0 = kb * 64 + ((pc ^ (i & 7)) << 3);
      if (row < a.vocab) src = a.head + (size_t)row * DM + k0;
    }
    out[id] = src ? *reinterpret_cast<const uint4*>(src) : make_uint4(0u, 0u, 0u, 0u);
  }
}

// cross-K/V [layer][B*S][K(DM) | V(DM)] -> [layer][image / 8][head][16-key chunk][image % 8][k|v][16 keys][32 channels] (blocks of 8
// images: the 16 KB a cluster pass needs per chunk and 8 images are contiguous), 16-byte chunk c of key r at chunk c ^ ((r >> 1) & 3);
// keys >= S and images >= B are zero rows (masked / never read)
__global__ void pack_cross_kv_kernel(const uint4* __restrict__ ckv, uint4* __restrict__ out, int B, int S, int nck, size_t n_chunks) {
  const int nb8 = (B + 7) >> 3;
  for (size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x; id < n_chunks; id += (size_t)gridDim.x * blockDim.x) {
    const size_t cell = id / 128; const int within = (int)(id % 128);        // 128 chunks of 16 bytes per 2 KB cell
    const int i8 = (int)(cell % 8), c = (int)((cell / 8) % nck), h = (int)((cell / (8 * (size_t)nck)) % CS);
    const size_t lb8 = cell / (8 * (size_t)nck * CS);                         // layer * nb8 + image block
    const int l = (int)(lb8 / nb8), b = (int)(lb8 % nb8) * 8 + i8;
    const int which = within / 64, r = (within % 64) / 4, pc = within % 4;
    const int key = c * 16 + r;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (key < S && b < B) v = ckv[((((size_t)l * B + b) * S + key) * (2 * DM) + which * DM + h * HD) / 8 + (pc ^ ((r >> 1) & 3))];
    out[id] = v;
  }
}

struct FusedCache {
  FusedParams P;
  bool valid;
};

bool geometry_ok(const mdc_dims& d) {
  if (d.precision != MDC_BF16 || d.dim != DM || d.dec_heads != CS || d.dec_ffn != FFN) return false;
  if (d.dec_layers < 1 || d.dec_layers > 8 || d.vocab > CS * VSL || d.vocab < 8) return false;
  if (d.n_patches < 1 || d.page_tokens != 16) return false;
  return true;
}

// ---- kernel variants --------------------------------------------------------------------------------------------------
// 0: NB = 1, 10-stage ring (160 KB), one CTA per SM   (<= 8 images per cluster; lowest latency of one batch)
// 1: NB = 2, 4-stage ring of 32 KB stages (128 KB), one CTA per SM    (<= 16 images per cluster)
// 2: NB = 1, 4-stage ring (64 KB), compact layout, two CTAs per SM (<= 8 images per cluster; two clusters interleave on the same SMs)
constexpr int N_VARIANTS = 3;
template <bool kTrace> struct Variants {
  template <bool kStop, bool kPrompt> static const void* fn_(int v) {
    switch (v) {
      case 0: return (const void*)decode_fused_kernel<kTrace, 1, 10, 1, kStop, kPrompt>;
      case 1: return (const void*)decode_fused_kernel<kTrace, 2, 4, 1, kStop, kPrompt>;
      default: return (const void*)decode_fused_kernel<kTrace, 1, 4, 2, kStop, kPrompt>;
    }
  }
  static const void* fn(int v, bool stop, bool prompt) {
    return prompt ? (stop ? fn_<true, true>(v) : fn_<false, true>(v)) : (stop ? fn_<true, false>(v) : fn_<false, false>(v));
  }
};
template <int NB, int NSTG, bool OVL> int lay_smem(bool prompt) { return prompt ? Lay<NB, NSTG, OVL>::SMEM_BYTES_PROMPT : Lay<NB, NSTG, OVL>::SMEM_BYTES; }
int variant_smem(int v, bool prompt) { return v == 0 ? lay_smem<1, 10, false>(prompt) : (v == 1 ? lay_smem<2, 4, true>(prompt) : lay_smem<1, 4, true>(prompt)); }

// per-context (= per-device) launch state: the dynamic-smem opt-in and the occupancy query are device properties
struct ClusterCtxState { int max_clusters[N_VARIANTS][2][2]; };      // [variant][stop at EOS][prompt]

}  // namespace

int decode_cluster_supported(const mdc_model* m, const mdc_decode_state* st, int t_end) {
  if (!geometry_ok(m->d) || !m->dec_pack) return 0;                // the packed weights are attached by mdc_decode_pack
  if (st->x_override || st->pos_override || st->per_op_kernels) return 0;
  if (t_end > 256 || st->pages_per_seq > 32 || st->n_pages < 1) return 0;
  return 1;
}

size_t decode_cluster_pack_bytes(const mdc_model* m) {
  if (!geometry_ok(m->d)) return 0;
  return (size_t)m->d.dec_layers * CS * BLOCKS_PER_LAYER * BLK_BYTES + (size_t)CS * HEAD_PACK_BYTES;
}

int decode_cluster_pack(mdc_model* m, void* out, cudaStream_t s) {
  const mdc_dims& d = m->d;
  const void** gw = m->w + MDC_ENC_GLOBAL_SLOTS + d.enc_depth * MDC_ENC_BLOCK_SLOTS;
  const void** lw0 = gw + MDC_DEC_GLOBAL_SLOTS;
  PackArgs a; memset(&a, 0, sizeof(a));
  for (int l = 0; l < d.dec_layers; ++l) {
    const void** lw = lw0 + l * MDC_DEC_LAYER_SLOTS;
    a.w[l][0] = (const __half*)lw[MDC_SA_IN_W]; a.w[l][1] = (const __half*)lw[MDC_SA_OUT_W]; a.w[l][2] = (const __half*)lw[MDC_CA_IN_W];
    a.w[l][3] = (const __half*)lw[MDC_CA_OUT_W]; a.w[l][4] = (const __half*)lw[MDC_FF1_W]; a.w[l][5] = (const __half*)lw[MDC_FF2_W];
  }
  a.head = (const __half*)gw[MDC_OUT_W]; a.layers = d.dec_layers; a.vocab = d.vocab;
  const size_t n = decode_cluster_pack_bytes(m) / 16;
  pack_weights_kernel<<<m->ctx->sm_count * 4, 256, 0, s>>>(a, (uint4*)out, n);
  MDC_LAUNCH_CHECK(m->ctx);
  m->dec_pack = out;
  if (m->fused_cache) ((FusedCache*)m->fused_cache)->valid = false;
  return 0;
}

// packed cross-K/V behind the plain [layer][B*S][2*DM] tensor in the caller's cross_kv buffer (mdc_cross_kv_bytes covers both)
size_t decode_cluster_ckv_pack_bytes(const mdc_model* m, int B) {
  if (!geometry_ok(m->d)) return 0;
  const int nck = (m->d.n_patches + 15) / 16;
  return (size_t)m->d.dec_layers * ((B + 7) / 8) * 8 * CS * nck * 2048;      // images padded to blocks of 8
}

int decode_cluster_ckv_pack(mdc_model* m, const void* ckv_plain, int B, void* out, cudaStream_t s) {
  const int S = m->d.n_patches, nck = (S + 15) / 16;
  const size_t n = decode_cluster_ckv_pack_bytes(m, B) / 16;
  pack_cross_kv_kernel<<<m->ctx->sm_count * 8, 256, 0, s>>>((const uint4*)ckv_plain, (uint4*)out, B, S, nck, n);
  MDC_LAUNCH_CHECK(m->ctx);
  return 0;
}

size_t decode_cluster_scratch_bytes(const mdc_model*, int) { return 0; }

void decode_cluster_model_destroy(mdc_model* m) {
  if (m && m->fused_cache) { delete (FusedCache*)m->fused_cache; m->fused_cache = nullptr; }
}

void decode_cluster_ctx_destroy(mdc_ctx* ctx) {
  if (ctx && ctx->decode_state) { delete (ClusterCtxState*)ctx->decode_state; ctx->decode_state = nullptr; }
}

int decode_cluster_launch(mdc_model* m, const mdc_decode_state* st, int t_begin, int t_end, void* /*logits_scratch*/, cudaStream_t s) {
  mdc_ctx* ctx = m->ctx; const mdc_dims& d = m->d;
  const void** gw = m->w + MDC_ENC_GLOBAL_SLOTS + d.enc_depth * MDC_ENC_BLOCK_SLOTS;
  const void** lw0 = gw + MDC_DEC_GLOBAL_SLOTS;
  if (!m->fused_cache) { FusedCache* c = new FusedCache(); memset(c, 0, sizeof(FusedCache)); m->fused_cache = c; }
  FusedCache* fc = (FusedCache*)m->fused_cache;
  if (!fc->valid) {
    FusedParams& P = fc->P;
    for (int l = 0; l < d.dec_layers; ++l) {
      const void** lw = lw0 + l * MDC_DEC_LAYER_SLOTS;
      P.b_in[l] = (const float*)lw[MDC_SA_IN_B]; P.b_so[l] = (const float*)lw[MDC_SA_OUT_B];
      P.ln1w[l] = (const float*)lw[MDC_LN1_W]; P.ln1b[l] = (const float*)lw[MDC_LN1_B];
      P.b_ca[l] = (const float*)lw[MDC_CA_IN_B]; P.b_co[l] = (const float*)lw[MDC_CA_OUT_B];
      P.ln2w[l] = (const float*)lw[MDC_LN2_W]; P.ln2b[l] = (const float*)lw[MDC_LN2_B];
      P.b_f1[l] = (const float*)lw[MDC_FF1_B]; P.b_f2[l] = (const float*)lw[MDC_FF2_B];
      P.ln3w[l] = (const float*)lw[MDC_LN3_W]; P.ln3b[l] = (const float*)lw[MDC_LN3_B];
    }
    P.wpack = (const uint8_t*)m->dec_pack;
    P.emb = (const float*)gw[MDC_EMB]; P.pos = (const float*)gw[MDC_DEC_POS]; P.b_out = (const float*)gw[MDC_OUT_B];
    P.layers = d.dec_layers; P.vocab = d.vocab; P.S = d.n_patches; P.pad_idx = d.pad_idx; P.PT = d.page_tokens;
    fc->valid = true;
  }
  FusedParams P = fc->P;
  P.B = st->B;
  P.tokens = st->tokens; P.tokens_ld = st->tokens_ld;
  P.kv_pool = (bf16*)st->kv_pool; P.page_table = st->page_table; P.pages_per_seq = st->pages_per_seq;
  P.logits_out = st->logits; P.logits_img_stride = (int64_t)st->logits_ld * d.vocab; P.logits_row_offset = st->logits_row_offset;
  P.confs = st->confs; P.confs_ld = st->confs_ld;
  P.uniforms = st->uniforms; P.uniforms_ld = st->uniforms_ld; P.top_k = st->top_k; P.top_p = st->top_p; P.forced = st->forced;
  P.eos = st->eos_token;
  P.prompt_len = st->prompt_len;
  P.t_begin = t_begin; P.t_end = t_end;
  P.trace = nullptr; P.trace_t = -1; P.ref_margin = 64.0f;
  int ipc = st->images_per_cluster, cps = st->ctas_per_sm;
#ifdef MDC_DEVTOOLS   // developer build only (tools/decode_trace.py): phase-trace buffer and variant overrides from the environment
  if (const char* tp = getenv("MDC_DECODE_TRACE_PTR")) { P.trace = (long long*)strtoull(tp, nullptr, 0); const char* tt = getenv("MDC_DECODE_TRACE_T"); P.trace_t = tt ? atoi(tt) : t_begin; }
  if (const char* e = getenv("MDC_DECODE_REF_MARGIN")) P.ref_margin = (float)atof(e);
  if (const char* e = getenv("MDC_DECODE_IPC")) ipc = atoi(e);
  if (const char* e = getenv("MDC_DECODE_CPS")) cps = atoi(e);
#endif
  P.ckv_pack = (const uint8_t*)st->cross_kv + align_up((size_t)d.dec_layers * st->B * d.n_patches * 2 * DM * 2, 256);
  // variant: more than 8 images per cluster -> the two-column-block instantiation; otherwise ctas_per_sm == 2 -> the compact one
  const int variant = ipc > 8 ? 1 : (cps == 2 ? 2 : 0);
  const int gmx = variant == 1 ? 16 : 8;
  if (!ctx->decode_state) { ClusterCtxState* cs = new ClusterCtxState(); memset(cs, 0, sizeof(*cs)); ctx->decode_state = cs; }
  ClusterCtxState* cs = (ClusterCtxState*)ctx->decode_state;
  const bool stop = st->stop_at_eos != 0, prompt = st->prompt_len != nullptr;
  const int smem = variant_smem(variant, prompt);
  if (!cs->max_clusters[variant][stop][prompt]) {
    const void* fn = Variants<false>::fn(variant, stop, prompt);
    MDC_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
#ifdef MDC_DEVTOOLS
    MDC_CUDA(cudaFuncSetAttribute(Variants<true>::fn(variant, stop, prompt), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
#endif
    cudaLaunchConfig_t q{}; q.gridDim = dim3(CS * 64); q.blockDim = dim3(NT); q.dynamicSmemBytes = smem;
    cudaLaunchAttribute a[1]; a[0].id = cudaLaunchAttributeClusterDimension; a[0].val.clusterDim.x = CS; a[0].val.clusterDim.y = 1; a[0].val.clusterDim.z = 1;
    q.attrs = a; q.numAttrs = 1;
    int n = 0;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&n, fn, &q);
    if (e != cudaSuccess || n < 1) { (void)cudaGetLastError(); n = ctx->sm_count / CS / 2; if (n < 1) n = 1; }
    cs->max_clusters[variant][stop][prompt] = n;
  }
  const int max_clusters = cs->max_clusters[variant][stop][prompt];
  int G = (P.B + max_clusters - 1) / max_clusters;
  if (ipc > 0 && ipc > G) G = ipc;                                                              // fewer, fuller clusters (batch pipelining)
  if (G > gmx) G = gmx;
  if (G < 1) G = 1;
  P.G = G;
  P.n_groups = (P.B + G - 1) / G;
  const int n_clusters = P.n_groups < max_clusters ? P.n_groups : max_clusters;
  void* args[1] = {(void*)&P};
  const void* fn = Variants<false>::fn(variant, stop, prompt);
#ifdef MDC_DEVTOOLS
  if (P.trace) fn = Variants<true>::fn(variant, stop, prompt);
#endif
  MDC_CUDA(cudaLaunchKernel(fn, dim3(n_clusters * CS), dim3(NT), args, (size_t)smem, s));
  MDC_LAUNCH_CHECK(ctx);
  return 0;
}
