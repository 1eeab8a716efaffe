"""Batch pipelining of the inference loop `for x in test_loader: generate(model, x, ...)` (inference_p.py:216-224).

One batch is two dependent phases with very different shapes on a B200:
  * encoder + cross-K/V build : ~90 short, wide kernels (tcgen05 GEMMs, strip attention) that fill all 148 SMs for ~2 ms
  * decode loop               : ONE persistent cluster kernel, latency-bound (a chain of dependent phases per layer), ~8-10 ms
Batches are independent (SURVEY 8e), so several are kept in flight: the encoder phase (and the host->device copy) of batch
i+1 runs on a low-priority stream WHILE the decode kernels of earlier batches run on high-priority streams.  For a single
batch the decode kernel spreads over as many 8-SM clusters as fit (13-15 x 5 images: lowest latency); in the pipeline it is
asked for 16 images per cluster instead (the kernel's two-column-block instantiation; 4 clusters = 32 SMs for B = 64: twice the
latency, but ~35 % less SM-time per batch), so that four decode kernels and an encoder share the 148 SMs.  Measured on B200
(tools/pipeline_probe.py, B=64, T=99, same box): serial 10.1 ms/batch; 8 images/cluster, 3 decode streams, 4 plans 6.91;
16 images/cluster with 3 streams / 6 plans 6.45, 4 / 6 6.11, 5 / 8 6.11 (saturated).
`depth` plans (static buffers + two CUDA graphs each) are used round-robin; events order encoder(i) -> decode(i) ->
encoder(i + depth).  Results are bit-identical to the serial `generate()`.
"""
from __future__ import annotations

import torch

from .inference import _check_bos, _host_result, _stop_token, _to_pinned, preprocess_bgr, preprocess_gray
from .model import GenerationPlan, check_max_len, replay


class Ticket:
    """Result handle of one submitted batch.  `tokens` / `confs` are device tensors valid in the order of `stream`;
    `result()` blocks the host until this batch (only) is done and returns the host copies."""

    def __init__(self, tokens, confs, host_tokens, host_confs, done, stream):
        self.tokens, self.confs = tokens, confs
        self._ht, self._hc, self._done, self.stream = host_tokens, host_confs, done, stream

    def result(self):
        self._done.synchronize()
        if self._ht is None:
            return self.tokens, self.confs
        return self._ht, self._hc


class GenerationPipeline:
    def __init__(self, model, batch, max_new_tokens, top_k=0, top_p=1.0, depth=None, decode_streams=None, images_per_cluster=16,
                 ctas_per_sm=0, to_host=False, device=None, eos_token=None):
        """`eos_token`: stop at that token, as EncoderDecoder.generate_tokens(..., eos_token=...) does."""
        if not hasattr(model, "_engine"):
            raise TypeError("GenerationPipeline needs the B200 EncoderDecoder; there is no PyTorch fallback path")
        eng = model._engine(device)
        T = int(max_new_tokens)
        check_max_len(T, eng.dims.max_pos)
        # operating point: the fused decode kernel holds 32 SMs for ~12 ms per batch -> 4 decode streams, 6 plans; geometries it does not
        # cover (dim 1024 of trail_01.py:158-160) decode as a chain of ~100 few-microsecond kernels per token on at most 64-192 CTAs,
        # which leaves most of the GPU idle per batch -> 8 decode streams, 10 plans (tools/config_t_probe.py: 720 -> 1 900 img/s)
        fused = getattr(eng, "dec_pack", None) is not None
        if decode_streams is None:
            decode_streams = 4 if fused else 8
        if depth is None:
            depth = 6 if fused else int(decode_streams) + 2
        self.eng, self.B, self.T, self.depth, self.to_host = eng, int(batch), T, int(depth), bool(to_host)
        dev = eng.device
        with torch.cuda.device(dev):
            self.plans = [GenerationPlan(eng, self.B, T, top_k, top_p, split=True, eos_token=eos_token,
                                         images_per_cluster=images_per_cluster, ctas_per_sm=ctas_per_sm) for _ in range(self.depth)]
            self.s_enc = torch.cuda.Stream(device=dev, priority=0)      # encoder / cross-K/V: fills whatever the decodes leave idle
            self.s_copy = torch.cuda.Stream(device=dev, priority=0)     # host->device copy (+ the u8 transform) of the NEXT batch: on the
            # encoder stream the 38.5 MB f32 copy of a batch (~0.8 ms on PCIe) sat between two encoder passes (e2e 4 % below the device-resident rate)
            self.copy_done = [torch.cuda.Event() for _ in range(self.depth)]
            self.enc_done = [torch.cuda.Event() for _ in range(self.depth)]
            self.dec_done = [torch.cuda.Event() for _ in range(self.depth)]
            self.s_decs = [torch.cuda.Stream(device=dev, priority=-1) for _ in range(max(1, int(decode_streams)))]   # clusters first
        self.n = 0

    def submit(self, image, uniforms=None):
        """image: f32 (B,3,H,W) on the device or in (pinned) host memory -- or raw u8 images, grayscale (B,h,w) or BGR (B,h,w,3) as
        cv2.imread returns them, which the fused preprocessing kernel (inference.preprocess_gray / preprocess_bgr: the reference's
        cv2-resize + normalise transform, bit-exact in its uint8 part) turns into the plan's input buffer on the device.
        Returns a Ticket."""
        i = self.n % self.depth
        p, busy = self.plans[i], self.n >= self.depth                   # busy: plan i has run before
        s_dec = self.s_decs[self.n % len(self.s_decs)]
        self.n += 1
        dev = self.eng.device
        gray = image.dtype == torch.uint8
        if gray:
            if image.dim() not in (3, 4) or image.shape[0] != self.B or (image.dim() == 4 and image.shape[-1] != 3):
                raise AssertionError("raw input must be uint8 (B,h,w) gray or (B,h,w,3) BGR")
        else:
            p.check_input(image)
        cur = torch.cuda.current_stream(dev)
        self.s_copy.wait_stream(cur)                                    # the caller's prior work on `image`
        with torch.cuda.stream(self.s_copy):
            if busy:
                self.s_copy.wait_event(self.enc_done[i])                # the plan's previous encoder pass has read its input buffer
            if gray:
                (preprocess_gray if image.dim() == 3 else preprocess_bgr)(image, size=p.x.shape[-1], out=p.x)
            else:
                p.x.copy_(image, non_blocking=True)
            self.copy_done[i].record(self.s_copy)
        self.s_enc.wait_stream(cur)
        with torch.cuda.stream(self.s_enc):
            if busy:
                self.s_enc.wait_event(self.dec_done[i])                 # plan buffers are free again
            self.s_enc.wait_event(self.copy_done[i])
            if p.uniforms is not None:
                if uniforms is None:
                    uniforms = torch.rand((self.B, self.T), dtype=torch.float32, device=dev)
                p.uniforms.copy_(uniforms.to(torch.float32), non_blocking=True)
            replay(dev, p.enc_graph)
            self.enc_done[i].record(self.s_enc)
        with torch.cuda.stream(s_dec):
            s_dec.wait_event(self.enc_done[i])
            replay(dev, p.dec_graph)
            tokens, confs = p.tokens.clone(), p.confs.clone()
            ht, hc = _to_pinned(tokens, confs) if self.to_host else (None, None)
            self.dec_done[i].record(s_dec)
            done = torch.cuda.Event()
            done.record(s_dec)
        return Ticket(tokens, confs, ht, hc, done, s_dec)

    def join(self):
        """Makes the caller's current stream wait for everything submitted so far (no host synchronisation)."""
        cur = torch.cuda.current_stream(self.eng.device)
        for sd in self.s_decs:
            cur.wait_stream(sd)
        cur.wait_stream(self.s_enc)
        cur.wait_stream(self.s_copy)


@torch.no_grad()
def generate_stream(model, batches, tokenizer, max_len=50, top_k=0, top_p=1, depth=None, stop_at_eos=False):
    """The reference's inference loop as ONE pipelined call: yields, per batch and in order, what `generate(model, x, tokenizer,
    max_len, top_k, top_p)` returns -- (LongTensor (B,1+max_len) on CPU, list of ceil(max_len/4) float tensors (B,) on CPU).
    `batches` is any iterable of f32 (B,3,H,W) tensors (host, ideally pinned, or device) -- or of raw grayscale u8 (B,h,w)
    tensors, normalised on the device (preprocess_gray).  `stop_at_eos`: as in generate()."""
    _check_bos(tokenizer)
    eos = _stop_token(tokenizer) if stop_at_eos else None
    pipes, pipe, pending = model.__dict__.setdefault("_stream_pipes", {}), None, []     # plans + graphs are reused across calls

    def finish(t):
        return _host_result(*t.result())

    for x in batches:
        dev = x.device if x.is_cuda else None
        key = ((x.shape[0], x.dim(), str(x.dtype)) if x.dtype == torch.uint8 else tuple(x.shape), int(max_len), int(top_k), float(top_p), depth, str(dev), eos)
        if key not in pipes or pipes[key].eng is not model._engine(dev):      # new shape (e.g. the ragged last batch) / new weights
            pipes[key] = GenerationPipeline(model, x.shape[0], max_len, top_k=top_k, top_p=top_p, depth=depth, to_host=True, device=dev,
                                            eos_token=eos)
        if pipes[key] is not pipe:
            while pending:                       # different plans share no events: drain before switching
                yield finish(pending.pop(0))
            pipe = pipes[key]
        pending.append(pipe.submit(x))
        if len(pending) > pipe.depth:            # keep `depth` batches in flight, hand out the oldest
            yield finish(pending.pop(0))
    while pending:
        yield finish(pending.pop(0))
