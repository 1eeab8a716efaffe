"""Token-id constants and the box/label part of the reference's token codec
(data_processing.py:224-290,317-391,556-598) -- the piece the hot path and its IoU stage need.

Sequence layout (data_processing.py:264-290):  BOS, <caption tokens>, label, xmin, ymin, xmax, ymax, EOS
with coordinate bins 0..num_bins-1, labels 258..267, UNK 299, BOS 300, EOS 301, PAD 302,
caption-start 303, caption-end 304, caption words from 270.  The spaCy vocabulary builder of the
reference is host-side data preparation and out of scope (SURVEY 2, `data_processing.py` row).
"""
from __future__ import annotations

import torch


def _select(logits, k, uniforms, want_prob):
    import ctypes as C  # noqa: F401
    from . import _lib as L
    from .config import CFG
    if logits.dim() != 2:
        raise ValueError("logits must be (batch, num_classes)")
    dev = logits.device if logits.is_cuda else torch.device(CFG.device)
    if dev.type != "cuda":
        raise L.MdcError("sampling runs on the GPU (mdc_select); there is no CPU fallback")
    lg = logits.to(dev, torch.float32).contiguous()
    B, V = lg.shape
    if uniforms is None:
        uniforms = torch.rand(B, device=dev)
    u = uniforms.to(dev, torch.float32).reshape(B).contiguous()
    tok = torch.empty(B, dtype=torch.int32, device=dev)
    prob = torch.empty(B, dtype=torch.float32, device=dev) if want_prob else None
    with torch.cuda.device(dev):
        L.check(L.lib().mdc_select(L.ctx(dev), L.ptr(lg), lg.stride(0), B, V, int(k), 1.0, L.ptr(u), L.ptr(tok), None, L.ptr(prob), L.stream_ptr()))
    return tok.long().view(B, 1), (prob.view(B, 1) if want_prob else None)


def top_k_sampling(logits, k, uniforms=None):
    """data_processing.py:786-790: keep the k largest logits (ties at the k-th kept), softmax, draw one index per row ->
    LongTensor (B,1).  The reference draws with torch.multinomial; here the draw is the inverse CDF of the same distribution at
    `uniforms` (B,) in [0,1) (torch.rand on the device when omitted), which makes it reproducible and testable against the
    oracle.  Unlike the reference the caller's `logits` tensor is not modified in place."""
    return _select(logits, k, uniforms, False)[0]


def top_k_sampling_with_scores_2d(logits, k, uniforms=None):
    """data_processing.py:803-835: as top_k_sampling, plus the sampled index's probability -> (LongTensor (B,1), f32 (B,1))."""
    return _select(logits, k, uniforms, True)


class Tokenizer:
    UNK_code, BOS_code, EOS_code, PAD_code = 299, 300, 301, 302
    CAPTION_START, CAPTION_END = 303, 304
    LABEL_BASE = 258

    def __init__(self, num_classes=10, num_bins=224, width=224, height=224, max_len=100, vocab=None):
        self.num_classes, self.num_bins = num_classes, num_bins
        self.width, self.height, self.max_len = width, height, max_len
        self.vocab = vocab                      # optional {id: word}
        self.vocab_size = 305 if vocab is None else max(305, max(vocab) + 1)

    def quantize(self, x):
        return (x * (self.num_bins - 1)).round().long()

    def dequantize(self, x):
        return x.float() / (self.num_bins - 1)

    # -- decode side: one kernel launch per batch (csrc/tokens.cu), no per-token host synchronisation ------------------
    def _grammar(self):
        from . import _lib as L
        g = L.TokenGrammar()
        g.pad, g.eos, g.caption_start, g.caption_end = self.PAD_code, self.EOS_code, self.CAPTION_START, self.CAPTION_END
        g.label_lo, g.label_hi = self.LABEL_BASE, self.LABEL_BASE + 9            # the reference's literal 258..267
        g.coord_max = 224                                                         # data_processing.py:583 literal bound
        g.num_bins, g.width, g.height = int(self.num_bins), int(self.width), int(self.height)
        return g

    def _run(self, mode, tokens, want_caption):
        """tokens: int (B,L) tensor (moved to CFG.device when it lives on the host).  Returns device tensors
        (boxes f32 (B,N,4), labels int32 (B,N), counts int32 (B,), caption int32 (B,L) | None, caption_len int32 (B,) | None)
        with N = (L+4)//5 rows (an upper bound of what either grammar can emit), rows >= counts zero."""
        import ctypes as C
        from . import _lib as L
        from .config import CFG
        if tokens.dim() == 1:
            tokens = tokens.unsqueeze(0)
        dev = tokens.device if tokens.is_cuda else torch.device(CFG.device)
        if dev.type != "cuda":
            raise L.MdcError("token decoding runs on the GPU (csrc/tokens.cu); there is no CPU fallback")
        t = tokens.to(dev, torch.int32).contiguous()
        B, Ln = t.shape
        N = max(1, (Ln + 4) // 5)
        boxes = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
        labels = torch.empty((B, N), dtype=torch.int32, device=dev)
        counts = torch.empty((B,), dtype=torch.int32, device=dev)
        cap = torch.empty((B, Ln), dtype=torch.int32, device=dev) if want_caption else None
        cap_len = torch.empty((B,), dtype=torch.int32, device=dev) if want_caption else None
        g = self._grammar()
        with torch.cuda.device(dev):
            L.check(L.lib().mdc_decode_tokens(L.ctx(dev), mode, L.ptr(t), t.stride(0), B, Ln, C.byref(g), N, L.ptr(labels), L.ptr(boxes),
                                              L.ptr(counts), L.ptr(cap), L.ptr(cap_len), L.stream_ptr()))
        return boxes, labels, counts, cap, cap_len

    def decode_bboxes(self, pred_seq):
        """data_processing.py:556-598: (B,L) tokens -> f32 (B, Nmax, 4) on the device, zero-row padded to the longest
        sequence of the batch (Nmax >= 1: an empty sequence is one zero box).  ONE launch + one scalar read (Nmax)."""
        from . import _lib as L
        boxes, _, counts, _, _ = self._run(L.TOK_BBOXES, torch.as_tensor(pred_seq), False)
        n = max(1, int(counts.max().item()))
        return boxes[:, :n].contiguous()

    def decode_bboxes_padded(self, pred_seq):
        """Sync-free form for pipelines (bench / parallel.pack_results): (boxes (B,N,4) with N = (L+4)//5, counts (B,))."""
        from . import _lib as L
        boxes, _, counts, _, _ = self._run(L.TOK_BBOXES, torch.as_tensor(pred_seq), False)
        return boxes, counts

    def caption_prompt(self, captions):
        """Prompts for caption-conditioned generation (generate(..., prompt=, prompt_lengths=)): a list of B caption-word-id lists ->
        (prompt LongTensor (B, P) with row b = [CAPTION_START, *captions[b], CAPTION_END] padded with PAD_code, lengths LongTensor (B,)),
        P the longest row.  Ids must be caption words, not special tokens."""
        rows = [[self.CAPTION_START, *[int(i) for i in ids], self.CAPTION_END] for ids in captions]
        if not rows:
            raise ValueError("caption_prompt needs at least one caption")
        special = {self.BOS_code, self.EOS_code, self.PAD_code, self.CAPTION_START, self.CAPTION_END}
        for b, r in enumerate(rows):
            if any(i in special or not 0 <= i < self.vocab_size for i in r[1:-1]):
                raise ValueError(f"caption {b} holds a special or out-of-vocabulary token id")
        P = max(len(r) for r in rows)
        prompt = torch.full((len(rows), P), self.PAD_code, dtype=torch.long)
        for b, r in enumerate(rows):
            prompt[b, :len(r)] = torch.tensor(r, dtype=torch.long)
        return prompt, torch.tensor([len(r) for r in rows], dtype=torch.long)

    def decode_batch(self, tokens):
        """Batched Tokenizer.decode (data_processing.py:317-391): device tensors (labels (B,N), boxes (B,N,4), counts (B,),
        caption ids (B,L) PAD-padded, caption lengths (B,), -1 = no caption markers)."""
        from . import _lib as L
        boxes, labels, counts, cap, cap_len = self._run(L.TOK_DECODE, torch.as_tensor(tokens), True)
        return labels, boxes, counts, cap, cap_len

    def tokens_to_text(self, ids):
        """data_processing.py:760-770 as `decode` uses it (a flat id list becomes one entry per token): list of words;
        `vocab` = {id: word} or an object with .itos."""
        table = getattr(self.vocab, "itos", self.vocab) or {}
        return [table.get(int(t), "<UNK>") for t in ids]

    def decode(self, tokens):
        """data_processing.py:317-391 for ONE sequence: (labels list, boxes list of [x0,y0,x1,y1], caption text)."""
        labels, boxes, counts, cap, cap_len = self.decode_batch(torch.as_tensor(tokens).reshape(1, -1))
        n, c = int(counts[0].item()), int(cap_len[0].item())
        text = "" if c < 0 else self.tokens_to_text(cap[0, :c].tolist())
        return labels[0, :n].tolist(), boxes[0, :n].double().tolist(), text
