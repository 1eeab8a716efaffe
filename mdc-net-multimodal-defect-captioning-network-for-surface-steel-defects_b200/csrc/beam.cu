// beam.cu -- beam-search bookkeeping between teacher-forced decode steps (mdc_beam_step / mdc_beam_finalize, include/mdc_b200.h).
// The decode kernels are not involved: a beam step runs after mdc_decode_steps(t, t+1) has written the step-t logits of the B*K rows.
//   beam_select_kernel   one CTA per image: log-softmax of each running beam's row, each beam's K best candidates (a warp per beam),
//                        the merge of the K*K candidates, then the reorder of token rows, scores, finish steps, per-token histories and
//                        the live page table (parents staged through the workspace first: a destination row can be another child's
//                        parent).  At a prompt step of its image (t + 1 <= prompt_len[b]) the CTA only records beam 0's zero log-prob
//                        and, when t % 4 == 0, its max probability, and marks every row as its own parent: nothing is selected or moved.
//   beam_kv_copy_kernel  copy-on-write of the partly filled KV page, twice: parents' valid token slots -> workspace, workspace -> each
//                        child's own page.  Skipped when the step filled its page (the page is then shared through the table), and
//                        for rows that are their own parent (kept places, prompt steps).
//   beam_finalize_kernel length-normalised scores (the length counts generated tokens only) and the best-first order of each image's
//                        beams.
#include "common.cuh"

namespace {

constexpr int BEAM_MAX_K = 16;
constexpr int BEAM_SEL_THREADS = BEAM_MAX_K * 32;
constexpr int BEAM_COPY_THREADS = 128;

struct BeamArgs {
  int B, K, V, pad, eos, pt, t, max_pos;
  const float* logits; int64_t logits_ld;
  int32_t* tokens; int32_t tokens_ld;
  const int32_t* prompt_len;           // int32 [B] or NULL
  int32_t* live; const int32_t* own; int32_t pps;
  float* scores; int32_t* finish;
  float* lps; int32_t lps_ld;
  float* confs; int32_t confs_ld;
  int32_t* parent;                     // workspace: parent row of each new row
  int32_t* stage_i; float* stage_f;    // workspace: staged parent token rows + page-table rows / log-prob + confidence rows
};

// workspace carve-up; the staged row prefixes are bounded by max_pos, the last step a decode can run
struct BeamWs { size_t parent, stage_i, stage_f, kv, total; int tok_w, pt_w, lp_w, cf_w; };

BeamWs beam_ws_layout(const mdc_dims& d, int B, int K, size_t page_bytes) {
  BeamWs w;
  const size_t BK = (size_t)B * K;
  w.tok_w = d.max_pos + 1; w.pt_w = (d.max_pos + d.page_tokens - 1) / d.page_tokens;
  w.lp_w = d.max_pos; w.cf_w = (d.max_pos + 3) / 4;
  w.parent = 0;
  w.stage_i = align_up(w.parent + BK * sizeof(int32_t), 256);
  w.stage_f = align_up(w.stage_i + BK * (w.tok_w + w.pt_w) * sizeof(int32_t), 256);
  w.kv = align_up(w.stage_f + BK * (w.lp_w + w.cf_w) * sizeof(float), 256);
  w.total = align_up(w.kv + BK * page_bytes, 256);
  return w;
}

// candidate order: higher score first, then lower token id (within one beam)
__device__ __forceinline__ bool cand_better(float c1, int v1, float c2, int v2) {
  if (v2 < 0) return v1 >= 0;
  if (v1 < 0) return false;
  return c1 > c2 || (c1 == c2 && v1 < v2);
}

__global__ void __launch_bounds__(BEAM_SEL_THREADS) beam_select_kernel(BeamArgs a) {
  __shared__ float c_score[BEAM_MAX_K * BEAM_MAX_K], c_lp[BEAM_MAX_K * BEAM_MAX_K];
  __shared__ int c_tok[BEAM_MAX_K * BEAM_MAX_K];
  __shared__ int s_fin[BEAM_MAX_K], s_win[BEAM_MAX_K];
  const int b = blockIdx.x, K = a.K, t = a.t, tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int64_t r0 = (int64_t)b * K;
  if (a.prompt_len && t < a.prompt_len[b]) {       // a prompt step of this image: column t+1 already holds the prompt token
    if (warp == 0) {
      if (a.confs && t % 4 == 0) {                  // beam 0's max probability 1 / sum exp(l - m), the quantity a greedy step reports
        const float* row = a.logits + r0 * a.logits_ld;
        float m = -INFINITY;
        for (int v = lane; v < a.V; v += 32) m = fmaxf(m, row[v]);
        m = warp_max(m);
        float sum = 0.f;
        for (int v = lane; v < a.V; v += 32) sum += expf(row[v] - m);
        sum = warp_sum(sum);
        if (lane == 0) a.confs[r0 * a.confs_ld + t / 4] = 1.f / sum;
      }
      if (lane == 0 && a.lps) a.lps[r0 * a.lps_ld + t] = 0.f;
    }
    if (tid < K) a.parent[r0 + tid] = (int32_t)(r0 + tid);   // the KV copy that follows moves nothing
    return;
  }
  if (tid < K) s_win[tid] = 0;        // fewer than K candidates only from a caller's state with no live beam: stay in bounds

  // 1. each beam's K best candidates, best first (a warp per beam)
  if (warp < K) {
    const int64_t r = r0 + warp;
    const float s = a.scores[r];
    const int f = a.finish[r];
    float* cs = c_score + warp * K; float* cl = c_lp + warp * K; int* ct = c_tok + warp * K;
    if (lane < K) ct[lane] = -1;
    if (lane == 0) s_fin[warp] = f;
    __syncwarp();
    if (f >= 0) {                                   // a finished beam has one candidate: PAD at an unchanged score
      if (lane == 0) { cs[0] = s; cl[0] = 0.f; ct[0] = a.pad; }
    } else if (s > -INFINITY) {
      const float* row = a.logits + r * a.logits_ld;
      float m = -INFINITY;
      for (int v = lane; v < a.V; v += 32) m = fmaxf(m, row[v]);
      m = warp_max(m);
      float sum = 0.f;                              // fixed order: lane-strided, then the xor tree (the same on every lane)
      for (int v = lane; v < a.V; v += 32) sum += expf(row[v] - m);
      sum = warp_sum(sum);
      const float lse = logf(sum);
      // K rounds of "the best candidate ordered after the previous pick": exact under ties, no exclusion mask
      float pc = INFINITY; int pv = -1;
      for (int i = 0; i < K; ++i) {
        float bc = -INFINITY, bl = 0.f; int bv = -1;
        for (int v = lane; v < a.V; v += 32) {
          const float lp = (row[v] - m) - lse;
          const float c = s + lp;
          const bool after = c < pc || (c == pc && v > pv);
          if (after && cand_better(c, v, bc, bv)) { bc = c; bl = lp; bv = v; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float oc = __shfl_xor_sync(0xffffffffu, bc, o), ol = __shfl_xor_sync(0xffffffffu, bl, o);
          const int ov = __shfl_xor_sync(0xffffffffu, bv, o);
          if (cand_better(oc, ov, bc, bv)) { bc = oc; bl = ol; bv = ov; }
        }
        if (lane == 0) { cs[i] = bc; cl[i] = bl; ct[i] = bv; }
        pc = bc; pv = bv;
      }
    }
  }
  __syncthreads();

  // 2. merge: the rank of each of the K*K candidates (higher score, then lower beam index, then lower token id)
  if (tid < K * K) {
    const int ti = c_tok[tid];
    if (ti >= 0) {
      const float ci = c_score[tid];
      const int ki = tid / K;
      int rank = 0;
      for (int j = 0; j < K * K; ++j) {
        const int tj = c_tok[j];
        if (tj < 0 || j == tid) continue;
        const float cj = c_score[j];
        const int kj = j / K;
        rank += (cj > ci || (cj == ci && (kj < ki || (kj == ki && tj < ti))));
      }
      if (rank < K) s_win[rank] = tid;
    }
  }
  __syncthreads();

  // 3. stage the parents' rows (known prefixes only)
  const int jc = t / a.pt;
  const int n_tok = t + 1, n_lp = t, n_cf = (t + 3) / 4, n_pt = jc + 1;
  const int wi = n_tok + n_pt, wf = n_lp + n_cf;
  const int tok_w = a.max_pos + 1, pt_w = (a.max_pos + a.pt - 1) / a.pt, lp_w = a.max_pos, cf_w = (a.max_pos + 3) / 4;
  for (int j = warp; j < K; j += BEAM_SEL_THREADS / 32) {
    const int64_t p = r0 + s_win[j] / K, r = r0 + j;
    if (lane == 0) a.parent[r] = (int32_t)p;
    int32_t* si = a.stage_i + r * (tok_w + pt_w);
    float* sf = a.stage_f + r * (lp_w + cf_w);
    for (int c = lane; c < wi; c += 32) si[c] = c < n_tok ? a.tokens[p * a.tokens_ld + c] : a.live[p * a.pps + (c - n_tok)];
    for (int c = lane; c < wf; c += 32)
      if (c < n_lp) { if (a.lps) sf[c] = a.lps[p * a.lps_ld + c]; }
      else if (a.confs) sf[c] = a.confs[p * a.confs_ld + (c - n_lp)];
  }
  __syncthreads();

  // 4. the new rows
  const bool page_full = (t % a.pt) == a.pt - 1;
  for (int j = warp; j < K; j += BEAM_SEL_THREADS / 32) {
    const int w = s_win[j], k = w / K;
    const int64_t r = r0 + j;
    const int fp = s_fin[k], v = c_tok[w];
    const float lp = fp >= 0 ? 0.f : c_lp[w];
    const int32_t* si = a.stage_i + r * (tok_w + pt_w);
    const float* sf = a.stage_f + r * (lp_w + cf_w);
    for (int c = lane; c < wi; c += 32) {
      if (c < n_tok) a.tokens[r * a.tokens_ld + c] = si[c];
      else {
        const int i = c - n_tok;
        a.live[r * a.pps + i] = (i < jc || page_full) ? si[c] : a.own[r * a.pps + i];
      }
    }
    for (int c = lane; c < wf; c += 32)
      if (c < n_lp) { if (a.lps) a.lps[r * a.lps_ld + c] = sf[c]; }
      else if (a.confs) a.confs[r * a.confs_ld + (c - n_lp)] = sf[c];
    if (lane == 0) {
      a.tokens[r * a.tokens_ld + t + 1] = v;
      if (a.lps) a.lps[r * a.lps_ld + t] = lp;
      if (a.confs && t % 4 == 0) a.confs[r * a.confs_ld + t / 4] = fp >= 0 ? 0.f : expf(lp);
      a.scores[r] = c_score[w];
      a.finish[r] = fp >= 0 ? fp : (v == a.eos ? t : -1);
    }
  }
}

// rows 0..n_tok-1 of every (layer, head, k|v) segment of one page: to_stage = 1 copies the parent's page jc (its own page: a partly
// filled page is never shared) into the row's workspace slot, 0 copies the slot into the row's own page jc.  Rows that kept their
// parent's place copy nothing.
__global__ void __launch_bounds__(BEAM_COPY_THREADS) beam_kv_copy_kernel(const int32_t* __restrict__ parent, const int32_t* __restrict__ own,
                                                                         int pps, int jc, uint8_t* pool, uint8_t* stage, int64_t page_bytes,
                                                                         int64_t seg_bytes, int copy_bytes, int n_seg, int to_stage) {
  const int64_t r = blockIdx.x;
  const int64_t p = parent[r];
  if (p == r) return;
  const uint8_t* src = to_stage ? pool + (int64_t)own[p * pps + jc] * page_bytes : stage + r * page_bytes;
  uint8_t* dst = to_stage ? stage + r * page_bytes : pool + (int64_t)own[r * pps + jc] * page_bytes;
  const int n16 = copy_bytes / 16;
  for (int s = blockIdx.y; s < n_seg; s += gridDim.y) {
    const uint4* sp = reinterpret_cast<const uint4*>(src + s * seg_bytes);
    uint4* dp = reinterpret_cast<uint4*>(dst + s * seg_bytes);
    for (int i = threadIdx.x; i < n16; i += BEAM_COPY_THREADS) dp[i] = sp[i];
  }
}

__global__ void beam_finalize_kernel(const float* __restrict__ scores, const int32_t* __restrict__ finish,
                                     const int32_t* __restrict__ prompt_len, int K, int T, float alpha, int32_t* __restrict__ order_out,
                                     float* __restrict__ norm_out) {
  __shared__ float s_norm[BEAM_MAX_K];
  const int b = blockIdx.x, k = threadIdx.x;
  float nk = 0.f;
  if (k < K) {
    const int f = finish[(int64_t)b * K + k];
    const int lb = prompt_len ? prompt_len[b] : 0;  // generated tokens only: the prompt columns are not part of the beam's length
    const float len = (float)((f >= 0 ? f + 1 : T) - lb);
    nk = scores[(int64_t)b * K + k] / powf(len, alpha);
    s_norm[k] = nk;
  }
  __syncthreads();
  if (k < K) {
    int rank = 0;
    for (int j = 0; j < K; ++j) rank += (s_norm[j] > nk || (s_norm[j] == nk && j < k));
    order_out[(int64_t)b * K + rank] = k;
    norm_out[(int64_t)b * K + rank] = nk;
  }
}

}  // namespace

extern "C" size_t mdc_beam_workspace_bytes(const mdc_model* m, int B, int K) {
  if (!m || B <= 0 || K < 1 || K > BEAM_MAX_K) return 0;
  return beam_ws_layout(m->d, B, K, mdc_kv_page_bytes(m)).total;
}

static int beam_check_state(const mdc_model* m, const mdc_beam_state* st) {
  MDC_CHECK_ARG(m && st && st->B > 0 && st->tokens && st->kv_pool && st->page_table && st->own_pages && st->scores &&
                st->finish_step && st->workspace);
  if (st->K < 1 || st->K > BEAM_MAX_K) MDC_FAIL(-2, "beam search: K = %d beams is outside 1..%d", st->K, BEAM_MAX_K);
  if (m->d.vocab > 4096) MDC_FAIL(-2, "beam search: vocabulary %d is larger than 4096", m->d.vocab);
  if (st->K > m->d.vocab) MDC_FAIL(-2, "beam search: K = %d beams exceeds the vocabulary %d", st->K, m->d.vocab);
  if (st->eos_token < 0 || st->eos_token >= m->d.vocab)
    MDC_FAIL(-2, "beam search: eos_token %d is outside the vocabulary [0, %d)", st->eos_token, m->d.vocab);
  const size_t need = mdc_beam_workspace_bytes(m, st->B, st->K);
  if (st->workspace_bytes < need)
    MDC_FAIL(-2, "beam search: workspace of %zu bytes is smaller than the %zu mdc_beam_workspace_bytes() requires", st->workspace_bytes, need);
  return 0;
}

extern "C" int mdc_beam_step(mdc_model* m, const mdc_beam_state* st, const float* logits, int64_t logits_ld, int t, void* stream) {
  MDC_TRY(beam_check_state(m, st));
  MDC_CHECK_ARG(logits && logits_ld >= m->d.vocab);
  MDC_CHECK_DEVICE(m->ctx);
  const mdc_dims& d = m->d;
  if (t < 0 || t >= d.max_pos || t + 1 >= st->tokens_ld || t >= st->pages_per_seq * d.page_tokens)
    MDC_FAIL(-2, "beam search: step %d is past the positional table (%d), the token columns (%d) or the pages (%d x %d tokens)",
             t, d.max_pos, st->tokens_ld, st->pages_per_seq, d.page_tokens);
  if (st->token_logprobs) MDC_CHECK_ARG(t < st->token_logprobs_ld);
  if (st->confs) MDC_CHECK_ARG(t / 4 < st->confs_ld);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t page_bytes = mdc_kv_page_bytes(m);
  const BeamWs w = beam_ws_layout(d, st->B, st->K, page_bytes);
  uint8_t* ws = (uint8_t*)st->workspace;
  BeamArgs a;
  a.B = st->B; a.K = st->K; a.V = d.vocab; a.pad = d.pad_idx; a.eos = st->eos_token; a.pt = d.page_tokens; a.t = t; a.max_pos = d.max_pos;
  a.logits = logits; a.logits_ld = logits_ld;
  a.tokens = st->tokens; a.tokens_ld = st->tokens_ld;
  a.prompt_len = st->prompt_len;
  a.live = st->page_table; a.own = st->own_pages; a.pps = st->pages_per_seq;
  a.scores = st->scores; a.finish = st->finish_step;
  a.lps = st->token_logprobs; a.lps_ld = st->token_logprobs_ld;
  a.confs = st->confs; a.confs_ld = st->confs_ld;
  a.parent = (int32_t*)(ws + w.parent); a.stage_i = (int32_t*)(ws + w.stage_i); a.stage_f = (float*)(ws + w.stage_f);
  beam_select_kernel<<<st->B, BEAM_SEL_THREADS, 0, s>>>(a);
  MDC_LAUNCH_CHECK(m->ctx);
  if (t % d.page_tokens != d.page_tokens - 1) {       // the page is partly filled: each moved beam copies it
    const int hd = d.dim / d.dec_heads, n_seg = d.dec_layers * d.dec_heads * 2;
    const int64_t seg_bytes = (int64_t)d.page_tokens * hd * esize(d.precision);
    const int copy_bytes = (t % d.page_tokens + 1) * hd * (int)esize(d.precision);
    const dim3 grid(st->B * st->K, n_seg < 65535 ? n_seg : 65535);
    for (int to_stage = 1; to_stage >= 0; --to_stage) {
      beam_kv_copy_kernel<<<grid, BEAM_COPY_THREADS, 0, s>>>(a.parent, st->own_pages, st->pages_per_seq, t / d.page_tokens,
                                                             (uint8_t*)st->kv_pool, ws + w.kv, (int64_t)page_bytes, seg_bytes,
                                                             copy_bytes, n_seg, to_stage);
      MDC_LAUNCH_CHECK(m->ctx);
    }
  }
  return 0;
}

extern "C" int mdc_beam_finalize(mdc_model* m, const mdc_beam_state* st, int T, float length_penalty, int32_t* order_out,
                                 float* norm_scores_out, void* stream) {
  MDC_TRY(beam_check_state(m, st));
  MDC_CHECK_ARG(order_out && norm_scores_out && T >= 1 && T <= m->d.max_pos);
  MDC_CHECK_DEVICE(m->ctx);
  beam_finalize_kernel<<<st->B, 32, 0, (cudaStream_t)stream>>>(st->scores, st->finish_step, st->prompt_len, st->K, T, length_penalty,
                                                                order_out, norm_scores_out);
  MDC_LAUNCH_CHECK(m->ctx);
  return 0;
}
