"""`generate()` and `postprocess()` with the reference's signatures (inference_p.py:69-115; the same
text lives in inference_trail_after_good_map.py:26-76), driving the incremental B200 decode loop:
encoder once, cross-attention K/V once, one fused decode step per new token, NO host
synchronisation inside the loop (the reference re-runs the whole model and syncs every 4th step).

Reference defects handled as SURVEY 0.2 prescribes: Q2 (`top_k_top_p_filtering` no longer exists in
transformers; its semantics are implemented inside the select kernel), Q5 (next-token logits :=
predict(x, prefix)[:, L]), Q6 (max_len <= CFG.max_len-1), Q9 (encoder hoisted out of the loop).
"""
from __future__ import annotations

import torch

from .config import CFG
from .model import check_max_len


@torch.no_grad()
def generate(model, x, tokenizer, max_len=50, top_k=0, top_p=1, uniforms=None, stop_at_eos=False, prompt=None, prompt_lengths=None):
    """Returns (LongTensor (B, 1+max_len) on CPU, list of ceil(max_len/4) float tensors (B,) on CPU).

    `uniforms` (B, max_len) in [0,1) is an optional superset argument: the per-step uniform variates
    of the top-k/top-p sampler (inverse-CDF draw), so that sampling is reproducible; by default they
    are drawn with torch.rand on the device (the reference uses torch.multinomial, inference_p.py:74).
    `stop_at_eos` (superset argument): stop at tokenizer.EOS_code.  Everything up to and including each
    image's first EOS is bitwise the default result; after it the tokens are PAD and the confidences 0,
    and decoding ends once every image has finished -- postprocess() returns the same either way.
    `prompt` int (B,P) / `prompt_lengths` int (B,) (superset arguments): decode each image from BOS followed by its first l_b prompt
    tokens (default l_b = P), e.g. a caption from tokenizer.caption_prompt() for caption-conditioned detection.  max_len counts the
    prompt, the output keeps its shape, the prompt columns hold the prompt, and postprocess_with_captions() returns a prompted caption.
    PAD or tokenizer.EOS_code inside a prompt, tokens outside the vocabulary and lengths outside 0..min(P, max_len) raise ValueError;
    semantics in EncoderDecoder.generate_tokens and DESIGN.md §3.4d."""
    _check_bos(tokenizer)
    if not hasattr(model, "generate_tokens"):
        raise TypeError("generate() needs the B200 EncoderDecoder; there is no PyTorch fallback path")
    eos = _stop_token(tokenizer) if stop_at_eos else None
    kw = {}
    if prompt is not None or prompt_lengths is not None:
        kw = {"prompt": prompt, "prompt_lengths": prompt_lengths}
        if eos is None:
            _check_prompt_eos(prompt, prompt_lengths, int(tokenizer.EOS_code))
    tokens, confs = model.generate_tokens(x, max_len, top_k=top_k, top_p=top_p, uniforms=uniforms, eos_token=eos, **kw)
    host = _to_pinned(tokens, confs)
    torch.cuda.current_stream(tokens.device).synchronize()      # the ONE sync of the whole call
    return _host_result(*host)


@torch.no_grad()
def generate_beam(model, x, tokenizer, max_len=50, num_beams=4, length_penalty=1.0, prompt=None, prompt_lengths=None):
    """Beam search (superset function): returns exactly what generate() returns -- LongTensor (B, 1+max_len) and a list of
    ceil(max_len/4) (B,) confidence tensors, on CPU -- for each image's best beam by score / len^length_penalty, so that postprocess()
    and postprocess_with_captions() read it unchanged.  Beams end at tokenizer.EOS_code (the tokens after it are PAD, the confidences 0);
    there is no early exit once every beam has ended, and no sampling inside beams.
    `prompt` int (B,P) / `prompt_lengths` int (B,) (superset arguments): every beam of image b starts from BOS followed by its first
    l_b prompt tokens (default l_b = P), e.g. a caption from tokenizer.caption_prompt(); the search starts after the prompt, and scores
    and the length normalisation count generated tokens only.  max_len counts the prompt and must leave one free step (l_b <= max_len
    - 1); PAD or tokenizer.EOS_code inside a prompt and tokens outside the vocabulary raise ValueError.  Semantics: DESIGN.md §3.4c."""
    _check_bos(tokenizer)
    if not hasattr(model, "generate_beam_tokens"):
        raise TypeError("generate_beam() needs the B200 EncoderDecoder; there is no PyTorch fallback path")
    check_max_len(int(max_len), int(CFG.max_len) - 1, ValueError)      # generate_beam_tokens raises RuntimeError
    if not x.is_cuda:
        raise ValueError("generate_beam() takes the images on a CUDA device; there is no CPU fallback")
    eos = _stop_token(tokenizer)
    tokens, _, _, confs = model.generate_beam_tokens(x, max_len, num_beams, length_penalty, eos_token=eos, prompt=prompt,
                                                     prompt_lengths=prompt_lengths)
    host = _to_pinned(tokens[:, 0], confs[:, 0])
    torch.cuda.current_stream(tokens.device).synchronize()
    return _host_result(*host)


def _check_prompt_eos(prompt, prompt_lengths, eos):
    """The tokenizer's EOS never belongs in a prompt, also without stop_at_eos (generate_tokens checks its own default EOS)."""
    if prompt is None:
        return
    p = torch.as_tensor(prompt).cpu()
    n = p.shape[-1] if prompt_lengths is None else torch.as_tensor(prompt_lengths).cpu().long().view(-1, 1)
    if p.dim() == 2 and bool(((p == eos) & (torch.arange(p.shape[-1])[None, :] < n)).any()):
        raise ValueError(f"a prompt may not hold EOS ({eos})")


def _to_pinned(tokens, confs):
    """Pinned host copies of a call's device tokens and confidences, enqueued on the current stream: valid once the call has
    synchronised."""
    host = torch.empty(tokens.shape, dtype=torch.int32, pin_memory=True)
    host_c = torch.empty(confs.shape, dtype=torch.float32, pin_memory=True)
    host.copy_(tokens, non_blocking=True)
    host_c.copy_(confs, non_blocking=True)
    return host, host_c


def _host_result(host, host_c):
    """generate()'s result from the host copies: LongTensor (B, 1+max_len) and the list of the ceil(max_len/4) (B,) confidence columns."""
    return host.long(), [host_c[:, i].clone() for i in range(host_c.shape[1])]


def _check_bos(tokenizer):
    if int(getattr(tokenizer, "BOS_code", CFG.bos_idx)) != int(CFG.bos_idx):
        raise ValueError("tokenizer.BOS_code must equal CFG.bos_idx (model.py:117 reads the global)")


def _stop_token(tokenizer):
    """The stop token of `stop_at_eos`; finished rows are filled with CFG.pad_idx, so the tokenizer's PAD must be that token."""
    if int(getattr(tokenizer, "PAD_code", CFG.pad_idx)) != int(CFG.pad_idx):
        raise ValueError("stop_at_eos fills finished rows with CFG.pad_idx: tokenizer.PAD_code must equal it")
    return int(tokenizer.EOS_code)


def _preprocess_u8(img_u8, size, out, channels):
    from . import _lib as L
    size = int(size or CFG.img_size)
    dev = img_u8.device if img_u8.is_cuda else torch.device(CFG.device)
    if dev.type != "cuda":
        raise L.MdcError("image preprocessing runs on the GPU; there is no CPU fallback")
    want_dim = 3 if channels == 1 else 4
    if img_u8.dtype != torch.uint8 or img_u8.dim() != want_dim or (channels == 3 and img_u8.shape[-1] != 3):
        raise ValueError("expected a uint8 (B,h,w) gray batch" if channels == 1 else "expected a uint8 (B,h,w,3) BGR batch")
    g = img_u8.to(dev, non_blocking=True).contiguous()
    B, h, w = g.shape[:3]
    if out is None:
        out = torch.empty((B, 3, size, size), dtype=torch.float32, device=dev)
    fn = L.lib().mdc_preprocess_gray if channels == 1 else L.lib().mdc_preprocess_bgr
    with torch.cuda.device(dev):
        L.check(fn(L.ctx(dev), L.ptr(g), B, h, w, L.ptr(out), size, L.stream_ptr(dev)))
    return out


def preprocess_gray(gray_u8, size=None, out=None):
    """The reference's image transform for NEU-DET-style grayscale inputs as ONE kernel (inference_p.py:148-158 / dataset.py:109-113):
    cv2.imread of a gray file = 3 equal channels, A.Resize(size, size) = cv2.resize(uint8, INTER_LINEAR) -- fixed-point bilinear,
    ROUNDED TO uint8, reproduced bit for bit -- then A.Normalize with the ImageNet mean / std in float32.
    u8 (B,h,w) on the device (or pinned host: copied first) -> f32 (B,3,size,size).  40 KB per 200x200 image cross PCIe instead of
    602 KB of float pixels."""
    return _preprocess_u8(gray_u8, size, out, 1)


def preprocess_bgr(bgr_u8, size=None, out=None):
    """The same transform for colour inputs exactly as `cv2.imread(path)` returns them: u8 (B,h,w,3), channels B,G,R.  The kernel does
    the `[..., ::-1]` flip (inference_p.py:152), the uint8 cv2 resize and A.Normalize; output f32 (B,3,size,size), channels R,G,B."""
    return _preprocess_u8(bgr_u8, size, out, 3)


def _postprocess(batch_preds, batch_confs, tokenizer):
    """Shared body of postprocess / postprocess_with_captions: first EOS, the reference's `(EOS-1) % 5` sanity rule (Q12, kept
    verbatim), then Tokenizer.decode of every sample -- as one batched GPU scan (csrc/tokens.cu) when the tokenizer is the B200 one."""
    EOS_idxs = (batch_preds == tokenizer.EOS_code).float().argmax(dim=-1)
    invalid_idxs = ((EOS_idxs - 1) % 5 != 0).nonzero().view(-1)
    EOS_idxs[invalid_idxs] = 0
    all_bboxes, all_labels, all_captions, all_confs = [], [], [], []
    batched = None
    if hasattr(tokenizer, "decode_batch"):
        # ONE kernel launch + one device->host copy for the whole batch instead of a tokenizer.decode() call (with its own
        # .item() reads) per sample: decode() drops PADs and cuts at the first EOS itself, so decoding the full row equals
        # decoding batch_preds[i, :EOS_idx + 1]
        labels_d, boxes_d, counts_d, cap_d, cap_len_d = tokenizer.decode_batch(batch_preds)
        batched = (labels_d.cpu(), boxes_d.cpu(), counts_d.cpu().tolist(), cap_d.cpu(), cap_len_d.cpu().tolist())
    for i, EOS_idx in enumerate(EOS_idxs.tolist()):
        if EOS_idx == 0:
            all_bboxes.append(None); all_labels.append(None); all_captions.append(None); all_confs.append(None)
            continue
        if batched is not None:
            lab, box, cnt, cap, cap_len = batched
            n, c = cnt[i], cap_len[i]
            decoded = (lab[i, :n].tolist(), box[i, :n].double().tolist(), "" if c < 0 else tokenizer.tokens_to_text(cap[i, :c].tolist()))
        else:
            decoded = tokenizer.decode(batch_preds[i, :EOS_idx + 1])
        if len(decoded) == 3:
            labels, bboxes, captions = decoded
        else:                                   # caption-less tokenizer API of inference_p.py:108
            labels, bboxes = decoded
            captions = None
        confs = [round(batch_confs[j][i].item(), 3) for j in range(len(bboxes))]
        all_bboxes.append(bboxes); all_labels.append(labels); all_captions.append(captions); all_confs.append(confs)
    return all_bboxes, all_labels, all_captions, all_confs


def postprocess(batch_preds, batch_confs, tokenizer):
    """inference_p.py:93-115: returns THREE lists (all_bboxes, all_labels, all_confs) -- the call site at inference_p.py:225 unpacks
    `bboxes, labels, confs = postprocess(...)`.  Entries are None for sequences the reference's sanity rule rejects."""
    all_bboxes, all_labels, _, all_confs = _postprocess(batch_preds, batch_confs, tokenizer)
    return all_bboxes, all_labels, all_confs


def postprocess_with_captions(batch_preds, batch_confs, tokenizer):
    """inference_trail_after_good_map.py:50-76, the caption-aware twin: FOUR lists (all_bboxes, all_labels, all_captions, all_confs)."""
    return _postprocess(batch_preds, batch_confs, tokenizer)
