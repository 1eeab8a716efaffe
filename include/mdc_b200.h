/*
 * mdc_b200.h -- C ABI of the B200-native (sm_100a) MDC-Net inference hot path.
 *
 * The reference (ashys2012/MDC-Net...) is pure Python/PyTorch and has NO FFI of its own
 * (SURVEY.md section 8b); its boundary is the Python surface of model.py / axial_model.py /
 * iou_calcualtions.py / iou_bbox.py / inference_p.py.  The Python host layer in
 * mdc-net-..._b200/ mirrors that surface one-to-one and binds THIS library through ctypes;
 * each entry point below names the reference code it replaces (paths relative to the
 * reference tree).  INTEGRATION.md shows the ctypes stub a maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; mdc_last_error() gives the text
 *     (thread-local).  There is no CPU fallback: without a CUDA device every compute call fails.
 *   - no allocation inside: weights, activations, workspaces, KV pages and page tables are
 *     caller-owned DEVICE buffers (torch tensors on the Python side); sizes come from the
 *     *_workspace_bytes() queries.  Only mdc_ctx/mdc_model (small host structs + cached
 *     CUtensorMap descriptors) are heap objects.
 *   - everything is asynchronous on the cudaStream_t passed as `stream` (void* here so that the
 *     header needs no CUDA include); calls are capturable into a CUDA graph.
 *   - plain pointers and sizes only; no torch types.
 */
#ifndef MDC_B200_H
#define MDC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDC_ABI_VERSION 10

/* element types of activations / weights.  MDC_F16 (IEEE half) is the type of the decode-loop weights under precision MDC_BF16
 * (see the weight table) and of mdc_gemm's fp16 mode. */
enum { MDC_F32 = 0, MDC_BF16 = 1, MDC_F16 = 2 };

/* GEMM epilogues: D = epi(A[M,K] . W[N,K]^T) */
enum {
  MDC_EPI_BIAS = 0,       /* D = acc + bias                                  (attn.qkv, cross K/V in-proj) */
  MDC_EPI_BIAS_GELU = 1,  /* D = gelu_erf(acc + bias)                        (timm Mlp.fc1 + nn.GELU)       */
  MDC_EPI_BIAS_RELU = 2,  /* D = relu(acc + bias)                            (TransformerDecoderLayer.linear1) */
  MDC_EPI_LS_RESIDUAL = 3,/* R(f32,in place) += gamma * (acc + bias)         (attn.proj / mlp.fc2 + LayerScale + residual) */
  MDC_EPI_PATCH = 4       /* R(f32)[row + row/period + 1] = acc + bias + pos[row % period]
                             (patch_embed.proj + pos_embed, rows shifted past each image's cls slot) */
};

/* IoU modes */
enum {
  MDC_IOU_EPS = 0,     /* inter / (union + 1e-6)         iou_calcualtions.py:5-40  bbox_iou            */
  MDC_IOU_PLAIN = 1,   /* inter / union  (0/0 = NaN)     iou_bbox.py:3-43          calculate_iou       */
  MDC_IOU_NAN0 = 2,    /* inter / union, NaN -> 0        iou_calcualtions.py:78-105 (torchvision.box_iou + nan_to_num) */
  MDC_IOU_GIOU = 3     /* iou - (enclose-union)/enclose  iou_calcualtions.py:220-255 giou_pairwise     */
};

typedef struct mdc_ctx mdc_ctx;
typedef struct mdc_model mdc_model;

/* ---- library / context ------------------------------------------------------------------ */
int mdc_abi_version(void);
const char* mdc_last_error(void);
/* One context per device (and per host thread that drives it).  Caches TMA descriptors. */
int mdc_ctx_create(int device, mdc_ctx** out);
int mdc_ctx_destroy(mdc_ctx* ctx);
/* number of kernels this library has launched through `ctx` since creation (bench.py's gpu_launches) */
int64_t mdc_ctx_launch_count(const mdc_ctx* ctx);

/* ---- (a) dense contractions ---------------------------------------------------------------
 * Replaces every nn.Linear / Conv2d(k=s=16) on the path: timm patch_embed.proj, attn.qkv,
 * attn.proj, mlp.fc1/fc2 (reached from model.py:17-22), and MultiheadAttention in-proj of the
 * memory (torch functional.py multi_head_attention_forward, reached from model.py:110-113).
 *   A [M,K] row-major (lda elements), W [N,K] row-major (nn.Linear layout), bias f32 [N] or NULL.
 *   dtype: MDC_BF16 -> A,W bf16, tcgen05.mma kind::f16 with fp32 TMEM accumulators, TMA-fed;
 *          MDC_F16  -> A,W and D IEEE half on the same kernel (bias / bias+ReLU epilogues only: the decoder prefill);
 *          MDC_F32  -> A,W f32, FFMA with fp32 accumulation in K order (the token-exact path).
 *   D is `dtype` for BIAS/GELU/RELU; for LS_RESIDUAL / PATCH the output is the f32 stream R.
 *   aux0: gamma f32[N] (LS_RESIDUAL) or, for PATCH, the positional table: `period` rows of N f32 values with the
 *         row stride of the output, ldd (pos[p][c] at aux0[p * ldd + c]); period: PATCH only.
 *   Alignment: MDC_F32 needs A and W 16-byte aligned, MDC_BF16 on the FFMA kernel 8-byte aligned; the tensor-core kernel
 *   (MDC_BF16 with K, lda, ldw, N multiples of 8, and MDC_F16) needs A, W and D 16-byte aligned, ldd % 8 == 0, and for
 *   PATCH a 16-byte aligned aux0 and period >= 32.  Misaligned operands are rejected before any launch.
 */
int mdc_gemm(mdc_ctx* ctx, int dtype, int epilogue,
             const void* A, int64_t lda, const void* W, int64_t ldw,
             void* D, int64_t ldd, const float* bias, const float* aux0, int period,
             int M, int N, int K, void* stream);

/* ---- (b) strip attention --------------------------------------------------------------------
 * softmax(q k^T * scale) v over independent strips, un-masked.  One kernel for
 *   (i)   axial_model.py:28-40 AxialAttention (one strip = whole token sequence, scale 0.125),
 *   (ii)  timm Attention inside the ViT blocks (strip = 197 tokens, head_dim 64, scale 1/8),
 *   (iii) true row / column strips of a patch grid (strip_len 14, n_strips = B*14).
 * qkv: [n_strips*strip_len, 3*heads*head_dim] packed q|k|v (row stride ld_qkv), out:
 * [n_strips*strip_len, heads*head_dim].  qkv must be 16-byte aligned and ld_qkv a multiple of 8.
 * softmax_over_queries != 0 selects softmax over the query axis (AxialAttention.forward(axis=-2));
 * it stages a whole strip in shared memory: strip_len <= 128, head_dim <= 128 and
 * (n(n+1) + 3·n·head_dim)·4 bytes (n = strip_len) within the device's per-block limit (227 KB on
 * a B200: n = 128 allows head_dim <= 104).
 */
int mdc_strip_attention(mdc_ctx* ctx, int dtype, const void* qkv, int64_t ld_qkv, void* out, int64_t ld_out,
                        int n_strips, int strip_len, int heads, int head_dim, float scale,
                        int softmax_over_queries, void* stream);

/* LayerNorm over the last axis of an f32 matrix, output `out_dtype` (timm norm1/norm2).
 * x, w and b must be 16-byte aligned, cols and ldx multiples of 4; `out` may have any stride (element alignment only). */
int mdc_layernorm(mdc_ctx* ctx, const float* x, int64_t ldx, const float* w, const float* b, float eps,
                  void* out, int64_t ldo, int out_dtype, int rows, int cols, void* stream);

/* The reference's image transform (inference_p.py:148-158 VOCDatasetTest, dataset.py:109-113) as one kernel:
 *   cv2.imread(...)[..., ::-1] -> A.Resize(size, size) -> A.Normalize() -> FloatTensor.permute(2, 0, 1)
 * A.Resize on a uint8 image is cv2.resize(INTER_LINEAR): fixed-point bilinear interpolation whose result is ROUNDED TO uint8
 * before A.Normalize turns it into float32 -- reproduced bit for bit (pinned against cv2 outputs); A.Normalize is
 * (v - mean*255) * (1/(std*255)) in float32 with the ImageNet mean / std.
 *   mdc_preprocess_gray: u8 (B,h,w) single-channel images (cv2.imread of a gray file yields three equal channels)
 *   mdc_preprocess_bgr : u8 (B,h,w,3) interleaved B,G,R as cv2.imread returns them; output channel order R,G,B
 * out: f32 NCHW (B,3,size,size). */
int mdc_preprocess_gray(mdc_ctx* ctx, const uint8_t* gray, int B, int h, int w, float* out, int size, void* stream);
int mdc_preprocess_bgr(mdc_ctx* ctx, const uint8_t* bgr, int B, int h, int w, float* out, int size, void* stream);

/* F.interpolate(mode='linear', align_corners=False) of a (n_in, dim) table to (n_out, dim): model.py:64-68 */
int mdc_interp_rows(mdc_ctx* ctx, const float* in, int n_in, float* out, int n_out, int dim, void* stream);

/* ---- model handle ----------------------------------------------------------------------------
 * Geometry of Encoder (model.py:14-23), Decoder (model.py:26-56) and the globals the reference
 * reads from CFG (model.py:32,60,94,117; utils.py:29).
 */
typedef struct mdc_dims {
  int32_t precision;     /* MDC_F32 or MDC_BF16 */
  int32_t img_size, patch, in_chans;
  int32_t enc_dim, enc_depth, enc_heads, enc_mlp;   /* deit3_medium: 512, 12, 8, 2048 */
  int32_t n_patches;     /* (img_size/patch)^2 = Decoder encoder_length */
  int32_t dim;           /* Encoder out_dim == Decoder dim */
  int32_t dec_heads, dec_layers, dec_ffn, vocab;
  int32_t max_pos;       /* CFG.max_len - 1 rows of decoder_pos_embed */
  int32_t pad_idx, bos_idx;
  int32_t has_axial;     /* axial_model.Decoder.axial_attention present */
  int32_t page_tokens;   /* self-attention KV page size in tokens (16) */
} mdc_dims;

/* Weight table: device pointers in the order of enum mdc_weight_slot, per-layer slots repeated.
 * GEMM weights are `precision` typed [N,K]; everything else (biases, norms, gammas, positional tables, embedding, cls token) is
 * f32.  The library keeps the pointers, never copies.
 * Decode-loop weights, the ones the autoregressive loop re-reads every step: MDC_SA_IN_W, MDC_SA_OUT_W, rows [0,dim) of
 * MDC_CA_IN_W (the cross-attention query projection), MDC_CA_OUT_W, MDC_FF1_W, MDC_FF2_W and MDC_OUT_W.  They are f32 under
 * precision MDC_F32 and IEEE half (MDC_F16) under MDC_BF16: fp16 has the same footprint and tensor-core rate as bf16 but 3 more
 * mantissa bits, and rounding these weights to bf16 alone costs 1.4e-2 of the 2e-2 max-abs logit budget (tools/error_budget_cpu.py),
 * to fp16 2e-3.  Rows [dim,3dim) of MDC_CA_IN_W (cross K/V in-projection, a tcgen05 GEMM against the bf16 memory) stay `precision`
 * typed, like every other GEMM weight and the KV caches. */
enum mdc_enc_slot {  /* encoder globals */
  MDC_W_PATCH = 0, MDC_B_PATCH, MDC_CLS, MDC_POS, MDC_NORM_W, MDC_NORM_B, MDC_ENC_GLOBAL_SLOTS
};
enum mdc_enc_block_slot {  /* per ViT block, after the globals */
  MDC_N1_W = 0, MDC_N1_B, MDC_QKV_W, MDC_QKV_B, MDC_PROJ_W, MDC_PROJ_B, MDC_LS1,
  MDC_N2_W, MDC_N2_B, MDC_FC1_W, MDC_FC1_B, MDC_FC2_W, MDC_FC2_B, MDC_LS2, MDC_ENC_BLOCK_SLOTS
};
enum mdc_dec_slot {  /* decoder globals, after all encoder slots */
  MDC_EMB = 0, MDC_DEC_POS, MDC_ENC_POS, MDC_OUT_W, MDC_OUT_B, MDC_AX_QKV_W, MDC_AX_OUT_W, MDC_AX_OUT_B,
  MDC_DEC_GLOBAL_SLOTS
};
enum mdc_dec_layer_slot {  /* per decoder layer, after the decoder globals */
  MDC_SA_IN_W = 0, MDC_SA_IN_B, MDC_SA_OUT_W, MDC_SA_OUT_B, MDC_LN1_W, MDC_LN1_B,
  MDC_CA_IN_W, MDC_CA_IN_B, MDC_CA_OUT_W, MDC_CA_OUT_B, MDC_LN2_W, MDC_LN2_B,
  MDC_FF1_W, MDC_FF1_B, MDC_FF2_W, MDC_FF2_B, MDC_LN3_W, MDC_LN3_B, MDC_DEC_LAYER_SLOTS
};

/* With decoder layers, the decoder's head width (dim / dec_heads) must be 32, 64 or 128 and dim at most 1024: the widths the
 * decode kernels cover.  Any other geometry is rejected here, before anything runs. */
int mdc_model_create(mdc_ctx* ctx, const mdc_dims* dims, const void* const* weights, int n_weights,
                     mdc_model** out);
int mdc_model_destroy(mdc_model* m);
int mdc_model_num_weights(const mdc_dims* dims);

/* ---- encoder: Encoder.forward, model.py:21-23 (timm VisionTransformer + AdaptiveAvgPool1d) ---
 * image f32 NCHW (B,3,img,img) -> enc_out f32 (B,n_patches,dim)  [what Encoder.forward returns]
 *                               -> memory `precision` (B,n_patches,dim) = enc_out + encoder_pos_embed
 *                                  (model.py:103-105), either output may be NULL.
 */
size_t mdc_encode_workspace_bytes(const mdc_model* m, int B);
int mdc_encode(mdc_model* m, const float* image, int B, float* enc_out, void* memory,
               void* workspace, size_t workspace_bytes, void* stream);
/* memory from a caller-provided encoder_out (Decoder.forward/predict entry): mem = enc_out + enc_pos */
int mdc_memory_from_encoder_out(mdc_model* m, const float* enc_out, int B, void* memory, void* stream);

/* ---- (c) cross-attention K/V, once per image, HBM resident -----------------------------------
 * cross_kv[l][b*S+s][0:dim]=K, [dim:2dim]=V  (`precision`), from rows [dim:3dim] of
 * multihead_attn.in_proj_weight (torch functional.py in-proj packing q|k|v).  Where the fused decode kernel covers the
 * geometry the buffer also carries, behind that tensor, the same values re-arranged per (layer, image, head, 16-key chunk)
 * into contiguous 2 KB cells that the kernel fetches with one bulk copy each; mdc_cross_kv_bytes() covers both parts. */
size_t mdc_cross_kv_bytes(const mdc_model* m, int B);
int mdc_cross_kv_build(mdc_model* m, const void* memory, int B, void* cross_kv, void* stream);

/* ---- (c,d) autoregressive decode ---------------------------------------------------------------
 * State of one batch being decoded.  All device buffers caller-owned.
 *   tokens   int32 [B, tokens_ld]   column 0..t are known when step t runs; step t writes column t+1
 *   kv_pool  `precision` [n_pages][dec_layers][heads][2][page_tokens][head_dim]   paged self-attention cache, zero-initialised by
 *            the caller (n_pages: pool extent).  The K and V rows of one (page, layer, head) are contiguous; with 64-byte rows the
 *            16-byte chunk c of token r sits at chunk c ^ ((r >> 1) & 3).  Opaque to callers: only the library reads or writes it.
 *   page_table int32 [B, pages_per_seq]  physical page of logical page j of image b
 *   logits   f32 [B, logits_ld, vocab] or NULL: row (t+1) receives the step-t logits
 *            (= predict(x, prefix)[:, t+1], the reference's shifted layout, model.py:116-123)
 *   confs    f32 [B, confs_ld] or NULL: max softmax prob of steps with t % 4 == 0 at column t/4
 *            (inference_p.py:84-86)
 *   uniforms f32 [B, uniforms_ld] or NULL: u in [0,1) per (image, step) for top-k/top-p sampling
 *   scratch  decode workspace, mdc_decode_workspace_bytes()
 */
typedef struct mdc_decode_state {
  int32_t B;
  int32_t* tokens; int32_t tokens_ld;
  void* kv_pool; const int32_t* page_table; int32_t pages_per_seq; int32_t n_pages;
  const void* cross_kv;
  float* logits; int32_t logits_ld;
  int32_t logits_row_offset;        /* step t writes logits row t + offset: 1 = predict's shifted layout, 0 = forward's */
  float* confs; int32_t confs_ld;
  const float* uniforms; int32_t uniforms_ld;
  int32_t top_k; float top_p;       /* 0 / 1.0 = greedy argmax (first max index on ties) */
  int32_t forced;                   /* 1 = teacher-forced: never write tokens (predict/forward) */
  const float* pos_override;        /* optional (n,dim) positional table (interpolated, model.py:64-68) */
  const float* x_override;          /* optional (B, n, dim) pre-computed input embeddings incl. pos (axial path) */
  int32_t x_override_ld;            /* n */
  void* scratch; size_t scratch_bytes;
  int32_t images_per_cluster;       /* 0 = spread the batch over as many 8-SM clusters as fit (lowest latency of ONE batch); 1..16 =
                                       at least that many images per cluster, i.e. fewer SMs per batch, so that several batches in
                                       flight (pipeline.py) share the GPU; more than 8 selects the kernel instantiation with two
                                       8-image column blocks per cluster pass.  On the per-operation path (geometries outside the fused
                                       kernel) 16 and more = "SM-time over latency": every weight-streaming linear takes two row tiles per
                                       CTA.  Does not change results (bitwise). */
  int32_t ctas_per_sm;              /* 0 / 1 = one decode CTA per SM (deep TMA ring); 2 (with images_per_cluster <= 8) = the compact
                                       shared-memory layout that lets two clusters -- two independent image groups -- share each
                                       SM, so that one group's dependent phase chain fills the other's stalls.  Bitwise the same
                                       results. */
  int32_t per_op_kernels;           /* 1 = run every step as per-operation kernels (decode.cu: the path of the fp32 token-exact
                                       mode and of geometries the fused cluster kernel does not cover) even where the fused kernel
                                       applies -- the parity tests compare the two implementations on the same inputs. */
  int32_t stop_at_eos;              /* 1 = stop at EOS (0, the zero-initialised value, = run every step for every image).  Let e_b be the
                                       first step at which image b emits `eos_token` (an EOS among the known columns 1..t_begin counts as
                                       finished from the start).  Token columns 0..e_b+1 and the conf columns of steps <= e_b are bitwise
                                       what the same call without stopping writes; token columns e_b+2..t_end are pad_idx and the conf
                                       columns of steps > e_b are 0.0, written by the library whatever the buffers held.  An image that
                                       never emits EOS gets the no-stop result.  Decoding of a group of images ends once all of them have
                                       finished (the fused kernel: per cluster group; the per-operation kernels: once the whole batch has
                                       finished, the remaining launches return at entry).  Results stay batch-invariant.  Requires
                                       forced == 0 and logits == NULL (steps that do not run have no logits). */
  int32_t eos_token;                /* the stop token, in [0, vocab) (read only with stop_at_eos) */
  const int32_t* prompt_len;        /* int32 [B] or NULL (= no prompt).  Prompted decoding: row b knows columns 0..l_b (l_b = prompt_len[b]),
                                       column 0 BOS and columns 1..l_b the caller's prompt, written into `tokens` before the call.  Step t
                                       with t + 1 <= l_b is a prompt step: its input is column t and it writes KV position t as any step;
                                       its output column t+1 keeps the prompt token (never written) and that token is what later steps
                                       read; it is never counted as an EOS; its conf column (t % 4 == 0) receives the max probability of
                                       the (filtered) distribution at that step, as a teacher-forced step writes it.  Steps t >= l_b run
                                       as without a prompt.  With a prompt equal to the first l_b tokens an unprompted call generates,
                                       tokens and confs are bitwise that call's.  With stop_at_eos the PAD / 0 pre-fill leaves the prompt
                                       columns alone.  The prompt must hold no EOS (the host layer rejects one).  Requires forced == 0. */
} mdc_decode_state;

size_t mdc_decode_workspace_bytes(const mdc_model* m, int B);
/* Decode-loop weights (see the weight table) pre-arranged for the fused decode kernel: per (layer, cluster rank) the
 * 32-row blocks the kernel consumes, in consumption order, each stored as the exact shared-memory image its tensor-core
 * fragment loads expect -- one contiguous bulk copy per pipeline stage instead of per-row tensor-map traffic.
 * mdc_decode_pack_bytes() is 0 when the fused kernel does not cover the model's geometry (the per-operation kernels then
 * serve mdc_decode_steps).  `packed` is a caller-owned device buffer that must outlive the model; call once after
 * mdc_model_create (and again if the weight buffers are rewritten in place). */
size_t mdc_decode_pack_bytes(const mdc_model* m);
int mdc_decode_pack(mdc_model* m, void* packed, void* stream);
size_t mdc_kv_page_bytes(const mdc_model* m);
/* steps t = t_begin .. t_end-1, back to back on `stream`, no host synchronisation inside. */
int mdc_decode_steps(mdc_model* m, const mdc_decode_state* st, int t_begin, int t_end, void* stream);

/* ---- teacher-forced decoder pass over all positions at once (Decoder.forward model.py:58-88, Decoder.predict model.py:92-127) ----
 * tokens int32 [B, tokens_ld] (first n columns: the target sequence as the reference builds it -- BOS-prepended for forward, PAD-padded
 * to max_len-1 for predict); pos f32 [n, dim] positional rows (NULL = decoder_pos_embed, n <= max_pos; forward passes the
 * interpolated table, model.py:64-68); cross_kv from mdc_cross_kv_build.  Every layer runs over the B*n rows in parallel:
 * tcgen05 GEMMs on the fp16 decode-loop weights, causal self-attention with the reference's float PAD-key mask (+1.0, utils.py:26-30),
 * cross-attention over the resident cross-K/V, fused residual + LayerNorm; then the vocabulary head.
 * logits f32 [B, logits_ld, vocab]: row (i + row_offset) receives the logits of position i for i < n_out (predict: row_offset 1,
 * n_out n-1; forward: 0, n).  Covered: the bf16 path (fp16 decode-loop weights) at model widths 256 / 512 / 1024 with head widths
 * 32 / 64 / 128 (configs P and T).  mdc_decoder_prefill_workspace_bytes() is 0 when the geometry is not covered (fp32 precision, width 64,
 * ...): the caller then runs mdc_decode_steps in teacher-forced mode, which computes the same logits step by step. */
size_t mdc_decoder_prefill_workspace_bytes(const mdc_model* m, int B, int n);
int mdc_decoder_prefill(mdc_model* m, const int32_t* tokens, int tokens_ld, int B, int n, const float* pos, const void* cross_kv,
                        float* logits, int logits_ld, int row_offset, int n_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- prompt prefill: steps [0, n) of a decode state as one all-positions pass ------------------------------------------------------
 * Equivalent, up to rounding, to mdc_decode_steps(st, 0, n) when every row knows columns 1..n (prompt_len[b] >= n, or the columns are
 * otherwise known): the same layer chain as mdc_decoder_prefill over columns 0..n-1 of st->tokens, and in addition it writes KV positions
 * 0..n-1 of every layer into the rows' pages through st->page_table (in st->precision, the pool layout mdc_decode_steps reads), the
 * logits rows t + logits_row_offset of steps t < n when st->logits is set, and the conf columns t / 4 (t % 4 == 0, t < n) when st->confs
 * is set -- the max probability of the distribution filtered by st->top_k / st->top_p, as the decode select computes it.  It never writes
 * tokens.  Afterwards mdc_decode_steps(st, n, T) continues.  Not with forced, x_override or per-step stop state (stop_at_eos is honoured by
 * the continuing mdc_decode_steps call, whose known prefix then covers columns 1..n).
 * mdc_decode_prefill_workspace_bytes() is 0 where the prefill does not cover the geometry (fp32 precision, widths other than
 * 256 / 512 / 1024, head widths other than 32 / 64 / 128): callers then run the prompt steps with mdc_decode_steps. */
size_t mdc_decode_prefill_workspace_bytes(const mdc_model* m, int B, int n);
int mdc_decode_prefill_steps(mdc_model* m, const mdc_decode_state* st, int n, void* workspace, size_t workspace_bytes, void* stream);

/* ---- beam search over the paged KV cache ---------------------------------------------------------------------------------
 * B images, K beams (1 <= K <= 16).  Row r = b*K + k of every [B*K, ...] buffer is beam k of image b; each row keeps a score s_r and a
 * finish step f_r (-1 while running).  Start: every token row [BOS, PAD, ...], s = 0 for k = 0 and -inf otherwise, f = -1; the page
 * table equals own_pages.  Step t (t = 0 .. T-1): mdc_decode_steps(t, t+1) teacher-forced (forced = 1) over the B*K rows writes the
 * step-t logits l, then mdc_beam_step(t):
 *   lp_r[v] = (l_v - m) - log sum_u exp(l_u - m) in f32 (m = row max; accurate expf/logf, a fixed reduction order);
 *   candidates: every (r, v) of a running row with s_r > -inf, scored s_r + lp_r[v]; exactly (r, PAD) at s_r for a finished row;
 *   per image the K best are kept (ties: lower beam index k, then lower token id); new beam j (0 = best) takes the parent's token row
 *   with column t+1 = v, the parent's KV of positions 0..t, the new score, f = f_parent if the parent had finished, t if v == eos_token,
 *   else -1, and the parent's per-token histories plus this step's entries: log-prob lp (0 for a finished parent's PAD) at column t,
 *   confidence exp(lp) (0 for a finished parent) at column t/4 when t % 4 == 0.
 * A row's score is therefore, bit for bit, the f32 sum of its per-token log-probs in step order.  No early exit, no sampling.
 * KV pages: row r writes only its own page own_pages[r][t / page_tokens] at step t.  At the reorder after step t (jc = t / page_tokens)
 * entries i < jc of a new beam's live row are its parent's (full pages, never written again, shared); entry jc is the parent's too when
 * step t filled that page, and otherwise the beam's own page jc, into which the parent's valid token slots 0 .. t % page_tokens are
 * copied (every layer, head, K and V; only when the parent is another row).  Parents' rows and pages are staged through the workspace
 * first, because a destination can be another child's source.  Buffers never move, so a whole beam search captures as one CUDA graph.
 *   tokens       int32 [B*K, tokens_ld]            the decode state's token rows (t + 1 < tokens_ld)
 *   kv_pool      the decode state's pool; page_table the live int32 [B*K, pages_per_seq] table mdc_decode_steps reads (rewritten here);
 *   own_pages    int32 [B*K, pages_per_seq] the rows' initial, distinct pages (never written)
 *   scores f32 [B*K], finish_step int32 [B*K]; token_logprobs f32 [B*K, token_logprobs_ld] and confs f32 [B*K, confs_ld], either NULL
 *   workspace    mdc_beam_workspace_bytes() (0 for K outside 1..16)
 * Prompted beam search (prompt_len int32 [B], NULL = no prompt): columns 1..l_b (l_b = prompt_len[b]) of all K token rows of image b
 * hold its prompt before step 0, and l_b <= T - 1 (at least one free step; the host layer checks it).  Step t with t + 1 <= l_b is a
 * prompt step of image b: its decode window reads column t as any step, and mdc_beam_step selects and reorders nothing for that image
 * -- beam 0 stays the only running beam at score 0, beams 1..K-1 stay at -inf, column t+1 keeps the prompt token, beam 0's log-prob
 * column t is 0 and, when t % 4 == 0, its conf column t/4 receives the max probability 1 / sum_u exp(l_u - m) of its distribution, as
 * a greedy prompt step writes it.  Prompt and free images mix within one step; each image's CTA decides alone.  The first free step
 * t = l_b is step 0 of an unprompted search: beam 0 is the only parent and its children take its KV through the reorder above.  Scores
 * count generated tokens only and stay the f32 sums of the per-token log-prob rows (prompt entries are 0).  With every l_b = 0 the
 * results are bitwise those of prompt_len = NULL.  Steps [0, n) with n <= min(l_b) may instead run as one mdc_decode_prefill_steps pass
 * over the B*K rows (confs set, no logits); the beam steps then start at t = n and the caller zeroes the log-prob columns t < n.
 * mdc_beam_finalize: normalised score s / len^length_penalty over the generated tokens, len = f + 1 - l_b for a finished beam and
 * T - l_b otherwise (l_b = 0 without a prompt); order_out int32 [B, K] lists each image's beam indices by normalised score, descending
 * (ties: lower index first), norm_scores_out f32 [B, K] in that order.
 * Rejected with a message: K outside 1..16 or above the vocabulary, vocab > 4096, eos_token outside the vocabulary, a t past the
 * positional table, the token columns or the pages, a short workspace. */
typedef struct mdc_beam_state {
  int32_t B, K;
  int32_t* tokens; int32_t tokens_ld;
  void* kv_pool; int32_t* page_table; const int32_t* own_pages; int32_t pages_per_seq;
  float* scores; int32_t* finish_step;
  float* token_logprobs; int32_t token_logprobs_ld;
  float* confs; int32_t confs_ld;
  int32_t eos_token;
  void* workspace; size_t workspace_bytes;
  const int32_t* prompt_len;        /* int32 [B] or NULL (= no prompt): see "Prompted beam search" above */
} mdc_beam_state;

size_t mdc_beam_workspace_bytes(const mdc_model* m, int B, int K);
/* selection, reorder and partial-page copy after step t: logits f32, row r's step-t logits at logits + r * logits_ld.  At most three
 * launches, no host synchronisation. */
int mdc_beam_step(mdc_model* m, const mdc_beam_state* st, const float* logits, int64_t logits_ld, int t, void* stream);
int mdc_beam_finalize(mdc_model* m, const mdc_beam_state* st, int T, float length_penalty, int32_t* order_out /*[B,K]*/,
                      float* norm_scores_out /*[B,K]*/, void* stream);

/* (d) head + select as a stand-alone op: logits f32 [B,V] -> token, max prob, probability of the selected token.
 * greedy: argmax(softmax(logits)) = first max index (inference_p.py:77);
 * top_k/top_p: transformers top_k_top_p_filtering (inference_p.py:83) then inverse-CDF draw with u.
 * Also serves data_processing.py:786-790 top_k_sampling and :803-835 top_k_sampling_with_scores_2d (prob_out = the sampled
 * token's softmax probability under the filtered distribution); any of the three outputs may be NULL. */
int mdc_select(mdc_ctx* ctx, const float* logits, int64_t ld, int B, int V, int top_k, float top_p,
               const float* uniforms, int32_t* token_out, float* conf_out, float* prob_out, void* stream);

/* AxialAttention.forward as a whole (axial_model.py:28-40): x f32 (B,n,dim) -> f32 (B,n,dim). */
size_t mdc_axial_workspace_bytes(const mdc_model* m, int B, int n);
int mdc_axial_attention(mdc_model* m, const float* x, int B, int n, int softmax_over_queries, float* out,
                        void* workspace, size_t workspace_bytes, void* stream);

/* axial_model.Decoder.forward front end (axial_model.py:100-103): out f32 (B,n,dim) =
 * AxialAttention(embedding[tokens]) + pos (pos NULL -> decoder_pos_embed, then n must equal max_pos). */
size_t mdc_axial_embed_workspace_bytes(const mdc_model* m, int B, int n);
int mdc_axial_embed(mdc_model* m, const int32_t* tokens, int tokens_ld, int B, int n, const float* pos,
                    int softmax_over_queries, float* out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- (e) batched box scores --------------------------------------------------------------------
 * pred f32 [B,N,4], gt f32 [B,M,4] xyxy, zero rows = padding (data_processing.py:596 pad_sequence).
 * iou_out f32 [B,N,M] or NULL; max_out f32 [B,N] row-max over GT or NULL (iou_calcualtions.py:59-75,
 * zero rows included, Q13).  One 128-bit load per box. */
int mdc_iou_batch(mdc_ctx* ctx, int mode, const float* pred, const float* gt, int B, int N, int M,
                  float* iou_out, float* max_out, void* stream);
/* giou_loss_with_scores (iou_calcualtions.py:165-208): per-image loss f32 [B] (zero-sum rows
 * filtered, penalty = #GT rows when nothing predicted) and the masked GIoU matrix f32 [B,N,M]
 * (NaN-free: entries of filtered rows/cols are written as 0 and flagged in valid u8 [B,N,M]). */
int mdc_giou_loss(mdc_ctx* ctx, const float* pred, const float* gt, int B, int N, int M, float no_detection_penalty,
                  float* loss_per_image, float* giou_out, uint8_t* valid_out, void* stream);

/* ---- detection metric: prediction <-> ground-truth matching ------------------------------------------------------------
 * The per-image greedy assignment behind mAP (reference: train_val_epoch.py:205-231, torchmetrics MeanAveragePrecision with
 * iou_thresholds = [0.3] -> pycocotools COCOeval.evaluateImg) for a batch in one launch: per image and class, detections in stable
 * descending score order (at most max_det per class); each takes the unmatched ground-truth box of its class with the highest
 * IoU >= iou_threshold.  pred_boxes f32 [B,N,4] xyxy, scores f32 [B,N], labels i32 [B,N], n_pred i32 [B] (valid rows per image);
 * gt_boxes f32 [B,M,4], gt_labels i32 [B,M], n_gt i32 [B].  N <= 128, M <= 128.
 * match_out i32 [B,N]: matched ground-truth index, -1 = false positive, -2 = not evaluated; order_out i32 [B,N]: position of the
 * detection in its image's score order (-1 = not evaluated).  The precision/recall accumulation over the whole set is host-side
 * (mdcnet_b200.metrics).  torchmetrics / pycocotools are absent here: restated from their published algorithm, parity unpinned. */
int mdc_map_match(mdc_ctx* ctx, const float* pred_boxes, const float* scores, const int32_t* labels, const int32_t* n_pred,
                  const float* gt_boxes, const int32_t* gt_labels, const int32_t* n_gt, int B, int N, int M, float iou_threshold,
                  int max_det, int32_t* match_out, int32_t* order_out, void* stream);

/* ---- token sequences -> labels / boxes / caption ids ---------------------------------------------------
 * The reference's per-sequence Python scans (with .item() syncs) between generate() and the IoU functions, as one launch.
 *   MDC_TOK_BBOXES  Tokenizer.decode_bboxes (data_processing.py:556-598): start after the first caption-end token (0 if none);
 *                   at a label token read the next four as a box, keep it when all are in [0,coord_max] and x1>x0, y1>y0,
 *                   advance 5 either way; stop at EOS; any other token advances 1; loop bound i < L-4.
 *   MDC_TOK_DECODE  Tokenizer.decode (data_processing.py:317-391), batched: PADs removed, cut at the first EOS, needs both
 *                   caption-start and caption-end; caption ids = the tokens between them; then fixed groups of five, kept when
 *                   the label is in range and all four values are in [0,coord_max].
 * De-quantisation: float32(v) / (num_bins-1) * width|height with the reference's two float32 roundings (:258-262, :551-553).
 * tokens int32 [B, tokens_ld] (first L columns used).  Outputs (device, caller-owned): boxes f32 [B,max_boxes,4] xyxy, rows
 * >= counts[b] zero (= pad_sequence's padding / the (1,4) zero box of an empty sequence); labels int32 [B,max_boxes] or NULL;
 * counts int32 [B]; caption int32 [B,L] padded with `pad` and caption_len int32 [B] (MDC_TOK_DECODE; may be NULL;
 * -1 = no caption-start/caption-end pair, for which the reference returns "" rather than a word list). */
enum { MDC_TOK_BBOXES = 0, MDC_TOK_DECODE = 1 };
typedef struct mdc_token_grammar {
  int32_t pad, eos, caption_start, caption_end;   /* 302, 301, 303, 304 (data_processing.py:235-239) */
  int32_t label_lo, label_hi;                     /* 258, 267 */
  int32_t coord_max;                              /* 224: the reference's literal bound (bins are 0..223) */
  int32_t num_bins, width, height;                /* 224, CFG.img_size, CFG.img_size */
} mdc_token_grammar;
int mdc_decode_tokens(mdc_ctx* ctx, int mode, const int32_t* tokens, int64_t tokens_ld, int B, int L,
                      const mdc_token_grammar* grammar, int max_boxes, int32_t* labels_out, float* boxes_out,
                      int32_t* counts_out, int32_t* caption_out, int32_t* caption_len_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MDC_B200_H */
