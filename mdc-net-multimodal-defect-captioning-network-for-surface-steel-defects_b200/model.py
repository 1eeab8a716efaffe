"""Host-side mirror of the reference's model.py: `Encoder`, `Decoder`, `EncoderDecoder` with the
same constructors, `forward()` / `predict()` semantics and state-dict keys (SURVEY.md 8b), but
every tensor operation runs in libmdc_b200.so (hand-written sm_100a kernels) through ctypes.

The nn.Modules here are PARAMETER CONTAINERS: they own the weights (so `load_state_dict` of a
reference checkpoint works, inference_p.py:132) and never run torch math on the hot path.  There
is no CPU / eager fallback -- calling forward without the CUDA library or a B200 raises.

Reference: /root/reference/model.py:14-23 (Encoder), :26-127 (Decoder), :147-181 (EncoderDecoder).
"""
from __future__ import annotations

import ctypes as C
import math
import os

import torch
from torch import nn

from . import _lib as L
from .config import CFG
from .kvcache import PagedKVCache

# timm model family table (embed_dim, depth, heads); the reference uses deit3_medium (allied_files.py:27)
_VIT_FAMILY = {
    "deit3_small_patch16_224": (384, 12, 6),
    "deit3_medium_patch16_224": (512, 12, 8),
    "deit3_base_patch16_224": (768, 12, 12),
    "deit3_large_patch16_224": (1024, 24, 16),
}


# ------------------------------------------------------------------------------------------------
# parameter containers with timm's key names (patch_embed.proj, blocks.i.{norm1,attn.qkv,attn.proj,
# ls1.gamma,norm2,mlp.fc1,mlp.fc2,ls2.gamma}, norm, cls_token, pos_embed)
# ------------------------------------------------------------------------------------------------
class _Holder(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("parameter container: the computation runs in libmdc_b200.so")


class _PatchEmbed(_Holder):
    def __init__(self, in_chans, dim, patch):
        super().__init__()
        self.proj = nn.Conv2d(in_chans, dim, kernel_size=patch, stride=patch)


class _Attn(_Holder):
    def __init__(self, dim):
        super().__init__()
        self.qkv = nn.Linear(dim, dim * 3, bias=True)
        self.proj = nn.Linear(dim, dim)


class _Mlp(_Holder):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)


class _Gamma(_Holder):
    def __init__(self, dim, init):
        super().__init__()
        self.gamma = nn.Parameter(init * torch.ones(dim))


class _Block(_Holder):
    def __init__(self, dim, init_values):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-6)
        self.attn = _Attn(dim)
        self.ls1 = _Gamma(dim, init_values)
        self.norm2 = nn.LayerNorm(dim, eps=1e-6)
        self.mlp = _Mlp(dim, dim * 4)
        self.ls2 = _Gamma(dim, init_values)


class VisionTransformerParams(_Holder):
    """DeiT-III ViT weights (timm `VisionTransformer`, no_embed_class=True, LayerScale 1e-6)."""

    def __init__(self, img_size=224, patch=16, in_chans=3, dim=512, depth=12, heads=8):
        super().__init__()
        self.img_size, self.patch, self.in_chans = img_size, patch, in_chans
        self.embed_dim, self.depth, self.num_heads = dim, depth, heads
        n = (img_size // patch) ** 2
        self.patch_embed = _PatchEmbed(in_chans, dim, patch)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, n, dim))
        self.blocks = nn.ModuleList([_Block(dim, 1e-6) for _ in range(depth)])
        self.norm = nn.LayerNorm(dim, eps=1e-6)
        nn.init.trunc_normal_(self.pos_embed, std=.02)
        nn.init.normal_(self.cls_token, std=1e-6)
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.trunc_normal_(m.weight, std=.02)
                nn.init.zeros_(m.bias)


# Decode-kernel launch options (mdc_decode_state.images_per_cluster / ctas_per_sm / per_op_kernels).  None of them changes a
# result bit (tests/test_gpu_model.py); they trade latency of one batch against SM-time per batch, and `per_op_kernels` lets the
# parity tests run the per-operation kernels where the fused cluster kernel would be picked; `prefill` = False makes
# forward() / predict() run the autoregressive kernels teacher-forced, step by step, instead of the all-positions prefill pass.
_DECODE_OPTIONS = {"images_per_cluster": 0, "ctas_per_sm": 0, "per_op_kernels": False, "prefill": True}


class decode_options:
    """`with decode_options(images_per_cluster=16): ...` -- scoped override of the decode launch options."""

    def __init__(self, **kw):
        bad = set(kw) - set(_DECODE_OPTIONS)
        if bad:
            raise TypeError(f"unknown decode option(s) {sorted(bad)}")
        self.kw, self.saved = kw, None

    def __enter__(self):
        self.saved = dict(_DECODE_OPTIONS)
        _DECODE_OPTIONS.update(self.kw)
        return self

    def __exit__(self, *exc):
        _DECODE_OPTIONS.clear(); _DECODE_OPTIONS.update(self.saved)
        return False


def _decode_options_key():
    return tuple(sorted((k, int(v)) for k, v in _DECODE_OPTIONS.items()))


def _precision_dtype(precision):
    if precision in ("bf16", torch.bfloat16):
        return torch.bfloat16
    if precision in ("fp32", "f32", torch.float32):
        return torch.float32
    raise ValueError(f"precision must be 'bf16' or 'fp32', got {precision!r}")


# ------------------------------------------------------------------------------------------------
# engine: prepared weights + mdc_model handle for an (encoder, decoder) pair
# ------------------------------------------------------------------------------------------------
class Engine:
    """Owns the device copies the kernels read (bf16 copies of the GEMM weights on the fast path, the
    parameters themselves on the fp32 path) and the C-side model handle.  Rebuilt when the precision,
    device or any parameter version changes (e.g. after load_state_dict)."""

    def __init__(self, encoder, decoder, precision, device):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.MdcError("MDC-Net B200 engine needs a CUDA device; there is no CPU fallback")
        self.dtype = _precision_dtype(precision)
        self.code = L.dtype_code(self.dtype)
        self.lib = L.lib()
        self.ctx = L.ctx(self.device)
        self.encoder, self.decoder = encoder, decoder
        self.keep = []          # tensors whose storage the C side points into
        table = []

        def gw(p):  # GEMM weight: [N,K] in the compute dtype
            if p is None:
                table.append(0); return
            t = p.detach().to(self.device, self.dtype).contiguous()
            t = t.reshape(t.shape[0], -1)
            self.keep.append(t); table.append(t.data_ptr())

        # decode-loop weights (re-read every step): fp16 on the bf16 path -- same bytes and tensor-core rate, 3 more mantissa
        # bits (bf16 rounding of these matrices alone costs 1.4e-2 of the 2e-2 logit budget); f32 on the fp32 path
        loop_dt = torch.float16 if self.dtype == torch.bfloat16 else torch.float32

        def lw(p, mixed_rows=None):
            """[N,K] in the loop dtype; `mixed_rows` = n: rows [0,n) loop dtype, the rest compute dtype (16-bit buffer)."""
            w = p.detach().to(self.device, torch.float32)
            if loop_dt == torch.float32:
                t = w.contiguous()
            else:
                t = w.clamp(-65504.0, 65504.0).to(torch.float16).contiguous()
                if mixed_rows is not None:
                    t = t.view(torch.int16).clone()
                    t[mixed_rows:] = w[mixed_rows:].to(self.dtype).view(torch.int16)
            self.keep.append(t); table.append(t.data_ptr())

        def fw(p):  # everything else stays fp32
            if p is None:
                table.append(0); return
            t = p.detach().to(self.device, torch.float32).contiguous()
            self.keep.append(t); table.append(t.data_ptr())

        d = L.Dims()
        d.precision = self.code
        d.page_tokens = int(getattr(CFG, "kv_page_tokens", 16))
        d.pad_idx, d.bos_idx = int(CFG.pad_idx), int(CFG.bos_idx)
        if encoder is not None:
            v = encoder.model
            d.img_size, d.patch, d.in_chans = v.img_size, v.patch, v.in_chans
            d.enc_dim, d.enc_depth, d.enc_heads, d.enc_mlp = v.embed_dim, v.depth, v.num_heads, v.embed_dim * 4
            d.n_patches = (v.img_size // v.patch) ** 2
            d.dim = encoder.out_dim
            gw(v.patch_embed.proj.weight); fw(v.patch_embed.proj.bias); fw(v.cls_token); fw(v.pos_embed)
            fw(v.norm.weight); fw(v.norm.bias)
            for b in v.blocks:
                fw(b.norm1.weight); fw(b.norm1.bias); gw(b.attn.qkv.weight); fw(b.attn.qkv.bias)
                gw(b.attn.proj.weight); fw(b.attn.proj.bias); fw(b.ls1.gamma)
                fw(b.norm2.weight); fw(b.norm2.bias); gw(b.mlp.fc1.weight); fw(b.mlp.fc1.bias)
                gw(b.mlp.fc2.weight); fw(b.mlp.fc2.bias); fw(b.ls2.gamma)
        else:
            d.img_size, d.patch, d.in_chans = 16, 16, 3
            d.enc_dim, d.enc_depth, d.enc_heads, d.enc_mlp = 64, 0, 1, 256
            d.n_patches = 1
            table.extend([0] * len(L.ENC_GLOBAL))
        if decoder is not None:
            if encoder is not None and decoder.dim != encoder.out_dim:
                raise ValueError("Encoder out_dim must equal Decoder dim")
            d.dim = decoder.dim
            d.n_patches = decoder.encoder_length if encoder is None else d.n_patches
            if encoder is not None and decoder.encoder_length != d.n_patches:
                raise ValueError(f"Decoder encoder_length {decoder.encoder_length} != encoder patches {d.n_patches}")
            layers = decoder.decoder.layers
            d.dec_heads, d.dec_layers = decoder.num_heads, len(layers)
            d.dec_ffn, d.vocab = (layers[0].linear1.out_features if len(layers) else 8), decoder.vocab_size
            d.max_pos = decoder.decoder_pos_embed.shape[1]
            ax = getattr(decoder, "axial_attention", None)
            d.has_axial = 1 if ax is not None else 0
            fw(decoder.embedding.weight); fw(decoder.decoder_pos_embed); fw(decoder.encoder_pos_embed)
            lw(decoder.output.weight); fw(decoder.output.bias)
            gw(ax.to_qkv.weight if ax is not None else None)
            gw(ax.to_out.weight if ax is not None else None)
            fw(ax.to_out.bias if ax is not None else None)
            for l in layers:
                lw(l.self_attn.in_proj_weight); fw(l.self_attn.in_proj_bias)
                lw(l.self_attn.out_proj.weight); fw(l.self_attn.out_proj.bias)
                fw(l.norm1.weight); fw(l.norm1.bias)
                lw(l.multihead_attn.in_proj_weight, mixed_rows=decoder.dim); fw(l.multihead_attn.in_proj_bias)
                lw(l.multihead_attn.out_proj.weight); fw(l.multihead_attn.out_proj.bias)
                fw(l.norm2.weight); fw(l.norm2.bias)
                lw(l.linear1.weight); fw(l.linear1.bias); lw(l.linear2.weight); fw(l.linear2.bias)
                fw(l.norm3.weight); fw(l.norm3.bias)
        else:
            d.dim = d.dim or 32
            d.dec_heads, d.dec_layers, d.dec_ffn, d.vocab, d.max_pos = max(1, d.dim // 32), 0, 8, 1, 1
            table.extend([0] * len(L.DEC_GLOBAL))
        self.dims = d
        n = self.lib.mdc_model_num_weights(C.byref(d))
        assert n == len(table), (n, len(table))
        arr = (C.c_void_p * n)(*table)
        h = C.c_void_p()
        L.check(self.lib.mdc_model_create(self.ctx, C.byref(d), arr, n, C.byref(h)))
        self.handle = h
        # decode-loop weights pre-arranged for the fused decode kernel (one bulk copy per pipeline stage); 0 bytes = other geometry
        nb = self.lib.mdc_decode_pack_bytes(h)
        self.dec_pack = None
        if nb:
            self.dec_pack = torch.empty(nb, dtype=torch.uint8, device=self.device)
            with torch.cuda.device(self.device):
                L.check(self.lib.mdc_decode_pack(h, L.ptr(self.dec_pack), L.stream_ptr(self.device)))

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.mdc_model_destroy(self.handle)
        except Exception:
            pass

    # ---- building blocks -------------------------------------------------------------------
    def encode(self, image, want_enc_out=True, want_memory=True):
        """image f32 (B,3,H,W) on device -> (enc_out f32 (B,n,dim) | None, memory `dtype` (B,n,dim) | None)"""
        d = self.dims
        if image.dim() != 4 or image.shape[1] != d.in_chans or image.shape[2] != d.img_size or image.shape[3] != d.img_size:
            raise AssertionError("Input size doesn't match model")      # timm PatchEmbed's strict check
        image = image.to(self.device, torch.float32).contiguous()
        B = image.shape[0]
        ws_bytes = self.lib.mdc_encode_workspace_bytes(self.handle, B)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        enc_out = torch.empty((B, d.n_patches, d.dim), dtype=torch.float32, device=self.device) if want_enc_out else None
        memory = torch.empty((B, d.n_patches, d.dim), dtype=self.dtype, device=self.device) if want_memory else None
        with torch.cuda.device(self.device):      # the C side checks that the current device is the context's
            L.check(self.lib.mdc_encode(self.handle, L.ptr(image), B, L.ptr(enc_out), L.ptr(memory), L.ptr(ws), ws_bytes, L.stream_ptr(self.device)))
        return enc_out, memory

    def memory_from(self, encoder_out):
        d = self.dims
        encoder_out = encoder_out.to(self.device, torch.float32).contiguous()
        B = encoder_out.shape[0]
        if tuple(encoder_out.shape[1:]) != (d.n_patches, d.dim):
            raise ValueError(f"encoder_out must be (B,{d.n_patches},{d.dim})")
        memory = torch.empty((B, d.n_patches, d.dim), dtype=self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self.lib.mdc_memory_from_encoder_out(self.handle, L.ptr(encoder_out), B, L.ptr(memory), L.stream_ptr(self.device)))
        return memory

    def cross_kv(self, memory):
        B = memory.shape[0]
        nbytes = self.lib.mdc_cross_kv_bytes(self.handle, B)
        ckv = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self.lib.mdc_cross_kv_build(self.handle, L.ptr(memory), B, L.ptr(ckv), L.stream_ptr(self.device)))
        return ckv

    def decode(self, cross_kv, tokens, t_begin, t_end, *, max_tokens, forced, logits=None, logits_row_offset=0,
               confs=None, uniforms=None, top_k=0, top_p=1.0, pos_override=None, x_override=None, kv=None, scratch=None,
               images_per_cluster=None, ctas_per_sm=None, per_op_kernels=None, eos_token=None, prompt_len=None, prefill=0,
               prefill_ws=None):
        """Runs decode steps [t_begin, t_end) back to back on the current stream (no host sync).  `eos_token` (free-running only): stop
        at that token -- after an image's first EOS its token columns are PAD and its confidences 0, and decoding ends once every image
        has finished (mdc_decode_state.stop_at_eos).  `prompt_len` (free-running only): int32 (B,) device tensor; row b's columns
        1..prompt_len[b] of `tokens` hold its prompt, which the prompt steps keep (mdc_decode_state.prompt_len).  `prefill` = n > 0 (with
        t_begin 0 and `prefill_ws`, mdc_decode_prefill_workspace_bytes): steps [0, n) run as one all-positions pass
        (mdc_decode_prefill_steps), the rest step by step."""
        d = self.dims
        B = tokens.shape[0]
        assert tokens.dtype == torch.int32 and tokens.is_contiguous()
        if kv is None:
            kv = PagedKVCache(B, max_tokens, d.dec_layers, d.dim, d.page_tokens, self.dtype, self.device)
        if scratch is None:
            scratch = torch.empty(self.lib.mdc_decode_workspace_bytes(self.handle, B), dtype=torch.uint8, device=self.device)
        st = L.DecodeState()
        st.B = B
        st.tokens, st.tokens_ld = tokens.data_ptr(), tokens.shape[1]
        st.kv_pool, st.page_table, st.pages_per_seq = kv.pool.data_ptr(), kv.page_table.data_ptr(), kv.pages_per_seq
        st.n_pages = kv.pool.shape[0]
        st.cross_kv = cross_kv.data_ptr()
        if logits is not None:
            assert logits.dtype == torch.float32 and logits.is_contiguous()
            st.logits, st.logits_ld = logits.data_ptr(), logits.shape[1]
        st.logits_row_offset = logits_row_offset
        if confs is not None:
            st.confs, st.confs_ld = confs.data_ptr(), confs.shape[1]
        if uniforms is not None:
            st.uniforms, st.uniforms_ld = uniforms.data_ptr(), uniforms.shape[1]
        st.top_k, st.top_p = int(top_k), float(top_p)
        st.forced = 1 if forced else 0
        if pos_override is not None:
            st.pos_override = pos_override.data_ptr()
        if x_override is not None:
            st.x_override, st.x_override_ld = x_override.data_ptr(), x_override.shape[1]
        st.scratch, st.scratch_bytes = scratch.data_ptr(), scratch.numel()
        opt = _DECODE_OPTIONS
        st.images_per_cluster = int(opt["images_per_cluster"] if images_per_cluster is None else images_per_cluster)
        st.ctas_per_sm = int(opt["ctas_per_sm"] if ctas_per_sm is None else ctas_per_sm)
        st.per_op_kernels = int(opt["per_op_kernels"] if per_op_kernels is None else per_op_kernels)
        if eos_token is not None:
            st.stop_at_eos, st.eos_token = 1, int(eos_token)
        if prompt_len is not None:
            assert prompt_len.dtype == torch.int32 and prompt_len.shape == (B,)
            st.prompt_len = prompt_len.data_ptr()
        with torch.cuda.device(self.device):
            if prefill:
                assert t_begin == 0 and prefill <= t_end
                L.check(self.lib.mdc_decode_prefill_steps(self.handle, C.byref(st), int(prefill), L.ptr(prefill_ws), prefill_ws.numel(),
                                                          L.stream_ptr(self.device)))
                t_begin = int(prefill)
            L.check(self.lib.mdc_decode_steps(self.handle, C.byref(st), t_begin, t_end, L.stream_ptr(self.device)))
        return kv, scratch

    def interp_pos(self, pos, length):
        """F.interpolate(mode='linear', align_corners=False) of the positional table (model.py:64-68)."""
        n, dim = pos.shape[-2], pos.shape[-1]
        src = pos.detach().to(self.device, torch.float32).reshape(n, dim).contiguous()
        if length == n:
            return src
        out = torch.empty((length, dim), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self.lib.mdc_interp_rows(self.ctx, L.ptr(src), n, L.ptr(out), length, dim, L.stream_ptr(self.device)))
        return out


def _param_signature(*modules):
    sig = []
    for m in modules:
        if m is None:
            continue
        for p in m.parameters():
            sig.append((p.data_ptr(), p._version))
    return tuple(sig)


class _EngineOwner:
    """Mixin: lazily (re)builds the Engine for the current precision / device / parameter versions."""

    def _engine_for(self, encoder, decoder, device=None):
        precision = getattr(self, "precision", None) or getattr(CFG, "precision", "bf16")
        if device is None:
            p = next(iter((encoder or decoder).parameters()))
            device = p.device if p.device.type == "cuda" else CFG.device
        device = torch.device(device)
        if device.type != "cuda":
            raise L.MdcError("MDC-Net B200: model/inputs must be on a CUDA device; there is no CPU fallback")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        key = (str(_precision_dtype(precision)), str(device), int(CFG.pad_idx), int(CFG.bos_idx), _param_signature(encoder, decoder))
        cache = self.__dict__.setdefault("_engine_cache", {})
        if cache.get("key") != key:
            cache["engine"] = Engine(encoder, decoder, precision, device)
            cache["key"] = key
        return cache["engine"]

    def set_precision(self, precision):
        """'bf16' (tcgen05 fast path) or 'fp32' (token-exact path); applies to every sub-module that owns an engine."""
        _precision_dtype(precision)
        self.precision = precision
        if isinstance(self, nn.Module):
            for m in self.modules():
                if m is not self and isinstance(m, _EngineOwner):
                    m.precision = precision
        return self


# ------------------------------------------------------------------------------------------------
# public classes (reference names / signatures)
# ------------------------------------------------------------------------------------------------
class Encoder(nn.Module, _EngineOwner):
    """model.py:14-23.  `img_size` is a superset argument (SURVEY 8b) needed for 512x512 inputs."""

    def __init__(self, model_name="deit3_base_patch16_224", pretrained=False, out_dim=256, img_size=224):
        super().__init__()
        if pretrained:
            raise RuntimeError("pretrained timm weights are not available offline; load a state_dict instead")
        base = model_name.split(".")[0]
        if base not in _VIT_FAMILY:
            raise ValueError(f"unknown model_name {model_name!r}; known: {sorted(_VIT_FAMILY)}")
        dim, depth, heads = _VIT_FAMILY[base]
        self.model = VisionTransformerParams(img_size=img_size, dim=dim, depth=depth, heads=heads)
        self.out_dim = out_dim
        self.precision = None

    def forward(self, x):
        eng = self._engine_for(self, None, x.device if x.is_cuda else None)
        enc_out, _ = eng.encode(x, want_enc_out=True, want_memory=False)
        return enc_out


class Decoder(nn.Module, _EngineOwner):
    """model.py:26-127.  The nn.TransformerDecoder instance is only the weight container (identical
    parameter names and initialisation order to the reference)."""

    def __init__(self, vocab_size, encoder_length, dim, num_heads, num_layers):
        super().__init__()
        self.dim, self.vocab_size, self.encoder_length, self.num_heads = dim, vocab_size, encoder_length, num_heads
        self.embedding = nn.Embedding(vocab_size, dim)
        self.decoder_pos_embed = nn.Parameter(torch.randn(1, CFG.max_len - 1, dim) * .02)
        decoder_layer = nn.TransformerDecoderLayer(d_model=dim, nhead=num_heads)
        self.decoder = nn.TransformerDecoder(decoder_layer, num_layers=num_layers)
        self.output = nn.Linear(dim, vocab_size)
        self._extra_init()      # axial variant creates its AxialAttention here (same RNG order as axial_model.py:66)
        self.encoder_pos_embed = nn.Parameter(torch.randn(1, encoder_length, dim) * .02)
        self.precision = None
        self.init_weights()

    def _extra_init(self):
        pass

    def init_weights(self):
        for name, p in self.named_parameters():
            if "encoder_pos_embed" in name or "decoder_pos_embed" in name:
                continue
            if p.dim() > 1:
                nn.init.xavier_uniform_(p)
        nn.init.trunc_normal_(self.encoder_pos_embed, std=.02)
        nn.init.trunc_normal_(self.decoder_pos_embed, std=.02)

    # -- shared driver ------------------------------------------------------------------------
    def _run_forced(self, eng, memory, tokens_i32, n_steps, out_rows, row_offset, pos_override=None, x_override=None):
        """Teacher-forced logits of positions [0, n_steps) into rows [row_offset, row_offset + n_steps) of a (B, out_rows, V) tensor.
        Default: ONE pass over all positions (mdc_decoder_prefill: GEMMs over B*n rows + causal attention); where that does not
        cover the model (fp32 token-exact mode, other geometries, the axial front end's precomputed embeddings) or with
        decode_options(prefill=False): the autoregressive kernels, step by step, on the same tokens."""
        B, n = tokens_i32.shape
        ckv = eng.cross_kv(memory)
        logits = torch.empty((B, out_rows, self.vocab_size), dtype=torch.float32, device=eng.device)
        ws_bytes = 0
        if x_override is None and _DECODE_OPTIONS["prefill"] and not _DECODE_OPTIONS["per_op_kernels"]:
            ws_bytes = eng.lib.mdc_decoder_prefill_workspace_bytes(eng.handle, B, n)
        if ws_bytes:
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=eng.device)
            with torch.cuda.device(eng.device):
                L.check(eng.lib.mdc_decoder_prefill(eng.handle, L.ptr(tokens_i32), tokens_i32.shape[1], B, n, L.ptr(pos_override), L.ptr(ckv),
                                                    L.ptr(logits), out_rows, row_offset, n_steps, L.ptr(ws), ws_bytes, L.stream_ptr(eng.device)))
            return logits
        eng.decode(ckv, tokens_i32, 0, n_steps, max_tokens=max(n_steps, 1), forced=True, logits=logits,
                   logits_row_offset=row_offset, pos_override=pos_override, x_override=x_override)
        return logits

    def forward(self, encoder_out, tgt):
        """(B,L) -> (B,L+1,V): prepends BOS, interpolates the positional table (model.py:58-88)."""
        eng = self._engine_for(None, self, encoder_out.device if encoder_out.is_cuda else None)
        return self._forward_with(eng, eng.memory_from(encoder_out), tgt)

    def _forward_with(self, eng, memory, tgt):
        B = tgt.shape[0]
        bos = torch.full((B, 1), int(CFG.bos_idx), dtype=torch.int32, device=eng.device)
        tokens = torch.cat([bos, tgt.to(eng.device, torch.int32)], dim=1).contiguous()
        n = tokens.shape[1]
        pos = eng.interp_pos(self.decoder_pos_embed, n)
        return self._run_forced(eng, memory, tokens, n, n, 0, pos_override=pos)

    def predict(self, encoder_out, tgt):
        """(B,L), L <= max_len-1 -> (B,max_len-1,V) with row 0 == bos_idx and row t = logits after
        tokens 0..t-1 over the PAD-padded sequence (model.py:92-127)."""
        eng = self._engine_for(None, self, encoder_out.device if encoder_out.is_cuda else None)
        return self._predict_with(eng, eng.memory_from(encoder_out), tgt)

    def _predict_with(self, eng, memory, tgt):
        B, Lp = tgt.shape
        n = int(CFG.max_len) - 1
        if n != self.decoder_pos_embed.shape[1]:
            raise RuntimeError("CFG.max_len changed after Decoder() was built (pos-embed is sized from it, model.py:32)")
        if Lp > n:
            raise RuntimeError(f"prefix length {Lp} exceeds CFG.max_len-1 = {n} (model.py:93, Q6)")
        tokens = torch.full((B, n), int(CFG.pad_idx), dtype=torch.int32, device=eng.device)
        tokens[:, :Lp] = tgt.to(eng.device, torch.int32)
        logits = self._run_forced(eng, memory, tokens, n - 1, n, 1)
        logits[:, 0, :] = float(CFG.bos_idx)       # the reference's constant first row (model.py:117-123)
        return logits


class EncoderDecoder(nn.Module, _EngineOwner):
    """model.py:147-181 (3-arg) and axial_model.py:161-174 (2-arg)."""

    def __init__(self, encoder, decoder, patch_dropout_rate=0.02):
        super().__init__()
        self.encoder, self.decoder = encoder, decoder
        self.patch_dropout_rate = patch_dropout_rate
        self.precision = None

    def _engine(self, device=None):
        if self.precision is None and (self.encoder.precision or self.decoder.precision):
            self.precision = self.encoder.precision or self.decoder.precision
        return self._engine_for(self.encoder, self.decoder, device)

    def forward(self, image, tgt):
        if self.training:
            raise RuntimeError("the B200 path is inference-only (call model.eval()); training-time patch "
                               "dropout (model.py:158-172) is out of scope")
        eng = self._engine(image.device if image.is_cuda else None)
        _, memory = eng.encode(image.to(eng.device), want_enc_out=False, want_memory=True)
        return self.decoder._forward_with(eng, memory, tgt)

    def predict(self, image, tgt):
        eng = self._engine(image.device if image.is_cuda else None)
        _, memory = eng.encode(image.to(eng.device), want_enc_out=False, want_memory=True)
        return self.decoder._predict_with(eng, memory, tgt)

    # -- the fast path used by generate(): encode once, cross-K/V once, incremental decode ---------
    def _plan(self, eng, key, use_graph, make):
        """The cached plan of one call shape; `make(use_graph)` builds it on first use.  Every plan is dropped when the engine changes
        (new weights, precision or device).  `use_graph` None: capture CUDA graphs unless MDC_NO_GRAPH=1."""
        if use_graph is None:
            use_graph = os.environ.get("MDC_NO_GRAPH", "0") != "1"
        key = (*key, bool(use_graph), _decode_options_key())
        plans = self.__dict__.setdefault("_plans", {})
        if plans.get("eng") is not eng:
            plans.clear(); plans["eng"] = eng
        if key not in plans:
            plans[key] = make(use_graph)
        return plans[key]

    @torch.no_grad()
    def generate_tokens(self, image, max_new_tokens, top_k=0, top_p=1.0, uniforms=None, return_logits=False, use_graph=None,
                        eos_token=None, prompt=None, prompt_lengths=None):
        """Returns (tokens int32 (B,1+T) on device, confs f32 (B,ceil(T/4)) on device[, logits (B,T,V)]).
        The whole call (encoder, cross-K/V, T decode steps) is one CUDA graph replay per (B, T, sampler, stop token, prompt) shape.
        `eos_token`: stop at that token (superset argument).  Up to and including an image's first EOS the result is bitwise the
        no-stop result; after it the tokens are PAD and the confidences 0, and decoding ends once every image has finished.  Not
        with `return_logits` (steps that do not run have no logits; predict()/forward() serve that use).
        `prompt` int (B,P) and `prompt_lengths` int (B,), each in 0..P (default P): prompted decoding (superset arguments).  Row b
        decodes from BOS followed by prompt[b, :l_b]: token columns 1..l_b keep the prompt, the conf column of a prompt step t (t % 4
        == 0) holds the max probability of the (filtered) distribution at that step, and steps t >= l_b select and sample as without a
        prompt.  T counts the prompt (l_b <= T).  With a prompt equal to the first l_b tokens an unprompted call returns, the result is
        bitwise that call's.  PAD or EOS (`eos_token`, default the tokenizer's 301) among the first l_b tokens, tokens outside the
        vocabulary, l_b outside 0..P or above T are rejected with ValueError.  The prompt and its lengths are read on the host:
        device tensors cost one synchronisation.  Where the all-positions prefill covers the model, the first min(l_b) steps run as one
        pass when min(l_b) >= PREFILL_MIN_STEPS (not under decode_options(prefill=False)); its results equal the step path's up to
        rounding."""
        eng = self._engine(image.device if image.is_cuda else None)
        B, T = image.shape[0], int(max_new_tokens)
        check_max_len(T, eng.dims.max_pos)
        if eos_token is not None:
            if return_logits:
                raise ValueError("return_logits=True cannot be combined with eos_token: steps that do not run have no logits")
            eos_token = check_eos_token(eos_token, eng.dims.vocab)
        P = n_prefill = 0
        if prompt is not None or prompt_lengths is not None:
            prompt, lengths = check_prompt(prompt, prompt_lengths, B, T, eng.dims.vocab, DEFAULT_EOS if eos_token is None else eos_token)
            P = prompt.shape[1]
            n = int(lengths.min())
            if (n >= PREFILL_MIN_STEPS and _DECODE_OPTIONS["prefill"]
                    and eng.lib.mdc_decode_prefill_workspace_bytes(eng.handle, B, n)):
                n_prefill = n
        plan = self._plan(eng, (id(eng), B, T, int(top_k), float(top_p), bool(return_logits), eos_token, P, n_prefill), use_graph,
                          lambda graph: GenerationPlan(eng, B, T, top_k, top_p, return_logits, graph, eos_token=eos_token,
                                                       prompt_width=P, prefill=n_prefill))
        if plan.uniforms is not None and uniforms is None:
            uniforms = torch.rand((B, T), dtype=torch.float32, device=eng.device)
        if P:
            plan.set_prompt(prompt, lengths)
        tokens, confs, logits = plan.run(image, uniforms)
        if return_logits:
            return tokens.clone(), confs.clone(), logits.clone()
        return tokens.clone(), confs.clone()

    @torch.no_grad()
    def generate_beam_tokens(self, image, max_new_tokens, num_beams, length_penalty=1.0, *, eos_token, use_graph=None, prompt=None,
                             prompt_lengths=None):
        """Beam search (superset method; semantics in include/mdc_b200.h and DESIGN.md §3.4c).  Returns, on the device, each image's
        beams best first by length-normalised score: tokens int32 (B,K,1+T), normalised scores f32 (B,K), per-token log-probs f32
        (B,K,T) and confidences f32 (B,K,ceil(T/4)).  Tokens after a beam's EOS are PAD, with log-prob and confidence 0.  The whole
        call (encoder, cross-K/V for the B*K rows, T x (one teacher-forced decode step + one beam step), the final ordering) is one
        CUDA graph replay per (B, T, K, length penalty, stop token, prompt) shape.
        `prompt` int (B,P) and `prompt_lengths` int (B,), each in 0..P (default P): every beam of image b starts from BOS followed by
        prompt[b, :l_b].  Steps t < l_b select nothing: the prompt columns are kept, their log-probs are 0, and the conf column of such a
        step (t % 4 == 0) holds the max probability of beam 0's distribution.  Step l_b is the first beam step.  Scores and the length
        normalisation count generated tokens only (len = f + 1 - l_b for a beam that ended at step f, T - l_b otherwise).  T counts the
        prompt, and a beam search needs a free step: l_b <= T - 1.  PAD or `eos_token` among the first l_b tokens, tokens outside the
        vocabulary and lengths outside 0..min(P, T - 1) raise ValueError before any launch; the prompt is read on the host.  With every
        l_b = 0 the result is bitwise the unprompted one; with K = 1 the tokens are prompted greedy generate_tokens'.  Where the
        all-positions prefill covers the model, the first min(l_b) steps of the B*K rows run as one pass when min(l_b) >=
        PREFILL_MIN_STEPS (not under decode_options(prefill=False)); its results equal the step path's up to rounding."""
        eng = self._engine(image.device if image.is_cuda else None)
        B, T, K = image.shape[0], int(max_new_tokens), int(num_beams)
        if not 1 <= K <= 16:
            raise ValueError(f"num_beams {K} is outside 1..16")
        if T < 1:
            raise RuntimeError(f"max_len {T}: beam search needs at least one new token")
        check_max_len(T, eng.dims.max_pos)
        eos_token = check_eos_token(eos_token, eng.dims.vocab)
        P = n_prefill = 0
        if prompt is not None or prompt_lengths is not None:
            prompt, lengths = check_beam_prompt(prompt, prompt_lengths, B, T, eng.dims.vocab, eos_token)
            P = prompt.shape[1]
            n = int(lengths.min())
            if (n >= PREFILL_MIN_STEPS and _DECODE_OPTIONS["prefill"]
                    and eng.lib.mdc_decode_prefill_workspace_bytes(eng.handle, B * K, n)):
                n_prefill = n
        plan = self._plan(eng, ("beam", id(eng), B, T, K, float(length_penalty), eos_token, P, n_prefill), use_graph,
                          lambda graph: BeamPlan(eng, B, T, K, length_penalty, eos_token, graph, prompt_width=P, prefill=n_prefill))
        if P:
            plan.set_prompt(prompt, lengths)
        return tuple(o.clone() for o in plan.run(image))


def check_max_len(T, max_pos, error=RuntimeError):
    """Generation reads one row of the decoder's positional table per new token, and the table has max_pos = CFG.max_len-1 rows."""
    if T > max_pos:
        raise error(f"max_len {T} exceeds CFG.max_len-1 = {max_pos}: the positional table has no more rows "
                    "(reference fails at model.py:93, Q6)")


# EOS of the reference tokenizer (data_processing.py:235-239): never allowed inside a prompt
DEFAULT_EOS = 301
# prompted generation: the first min(l_b) steps run as one all-positions prefill pass from this many prompt steps on (DESIGN.md §3.4d)
PREFILL_MIN_STEPS = 6


def check_prompt(prompt, prompt_lengths, B, T, vocab, eos_token):
    """Host copies of a generation prompt, checked: (prompt int32 (B, min(P, T)) with PAD after each row's length, lengths int32 (B,))."""
    if prompt is None:
        raise ValueError("prompt_lengths needs a prompt")
    prompt = torch.as_tensor(prompt).detach().cpu()
    if prompt.dim() != 2 or prompt.shape[0] != B:
        raise ValueError(f"prompt must be (B, P) with B = {B} images, got {tuple(prompt.shape)}")
    if prompt.dtype.is_floating_point or prompt.dtype == torch.bool:
        raise ValueError("prompt must hold integer token ids")
    P = prompt.shape[1]
    if prompt_lengths is None:
        lengths = torch.full((B,), P, dtype=torch.int64)
    else:
        lengths = torch.as_tensor(prompt_lengths).detach().cpu()
        if lengths.shape != (B,) or lengths.dtype.is_floating_point or lengths.dtype == torch.bool:
            raise ValueError(f"prompt_lengths must be {B} integers")
        lengths = lengths.long()
    if bool((lengths < 0).any()) or bool((lengths > P).any()):
        raise ValueError(f"prompt_lengths must lie in 0..{P} (the prompt width), got {lengths.tolist()}")
    if bool((lengths > T).any()):
        raise ValueError(f"a prompt length exceeds max_len {T}: max_len counts the prompt")
    prompt = prompt.long()
    live = torch.arange(P)[None, :] < lengths[:, None]
    bad = live & ((prompt < 0) | (prompt >= vocab))
    if bool(bad.any()):
        raise ValueError(f"prompt tokens must lie in [0, {vocab}): row {int(bad.any(1).nonzero()[0])}")
    special = live & ((prompt == int(CFG.pad_idx)) | (prompt == int(eos_token)))
    if bool(special.any()):
        raise ValueError(f"a prompt may not hold PAD ({int(CFG.pad_idx)}) or EOS ({int(eos_token)}): row {int(special.any(1).nonzero()[0])}")
    W = min(P, T)
    out = torch.where(live, prompt, torch.full_like(prompt, int(CFG.pad_idx)))[:, :W]
    return out.to(torch.int32).contiguous(), lengths.to(torch.int32)


def check_beam_prompt(prompt, prompt_lengths, B, T, vocab, eos_token):
    """check_prompt, plus the rule of beam search: every prompt leaves at least one step to search (l_b <= T - 1)."""
    prompt, lengths = check_prompt(prompt, prompt_lengths, B, T, vocab, eos_token)
    if bool((lengths > T - 1).any()):
        raise ValueError(f"a prompt length exceeds max_len - 1 = {T - 1}: beam search needs at least one step after the prompt")
    return prompt, lengths


def check_eos_token(eos_token, vocab):
    eos_token = int(eos_token)
    if not 0 <= eos_token < vocab:
        raise ValueError(f"eos_token {eos_token} is outside the vocabulary [0, {vocab})")
    return eos_token


def capture_graphs(device, *launches):
    """Captures each of `launches` (functions that enqueue work on the current stream) into its own CUDA graph and returns, in the same
    order, (graph, kernels of libmdc_b200.so in one replay) pairs for replay().  All of them run once first as a warm-up (tensor maps,
    shared-memory attributes, lazy module load), then the device is synchronised.  Warm-up and capture run under `device`, on one side
    stream of it given explicitly: torch's default capture stream is a process-wide singleton on whichever device captured first, and a
    graph of another device captured there replays nothing."""
    with torch.cuda.device(device):
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            for launch in launches:
                launch()
        torch.cuda.current_stream(device).wait_stream(side)
        torch.cuda.synchronize(device)
        graphs = []
        for launch in launches:
            graph, n0 = torch.cuda.CUDAGraph(), L.launch_count(device)
            with torch.cuda.graph(graph, stream=side):
                launch()
            graphs.append((graph, L.launch_count(device) - n0))
        return graphs


def replay(device, captured):
    """Replays one (graph, kernel count) pair of capture_graphs() on the current stream and counts its kernels in L.launch_count."""
    graph, n_kernels = captured
    graph.replay()
    L.note_graph_replay(device, n_kernels)


class _Plan:
    """Static buffers of one generation call shape on the engine's device: the B input images `x`, the encoder workspace and `memory`,
    and for the `rows` decoded sequences (B, or B*K beams) the cross-K/V, tokens, confidences, KV cache and decode scratch.  A plan
    launches its whole call in `_launch` (no host synchronisation inside) and returns `_outputs()`; `run` replays `graph` instead
    where the plan captured one.  `uniforms`: the sampler's variates, for plans that sample."""

    graph = uniforms = None

    def __init__(self, eng, B, T, rows):
        d, dev = eng.dims, eng.device
        self.eng, self.B, self.T = eng, B, T
        self.x = torch.zeros((B, d.in_chans, d.img_size, d.img_size), dtype=torch.float32, device=dev)
        self.ws_bytes = eng.lib.mdc_encode_workspace_bytes(eng.handle, B)
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.memory = torch.empty((B, d.n_patches, d.dim), dtype=eng.dtype, device=dev)
        self.ckv = torch.empty(eng.lib.mdc_cross_kv_bytes(eng.handle, rows), dtype=torch.uint8, device=dev)
        self.tokens = torch.empty((rows, T + 1), dtype=torch.int32, device=dev)
        self.confs = torch.zeros((rows, (T + 3) // 4), dtype=torch.float32, device=dev)
        self.kv = PagedKVCache(rows, T, d.dec_layers, d.dim, d.page_tokens, eng.dtype, dev)
        self.scratch = torch.empty(eng.lib.mdc_decode_workspace_bytes(eng.handle, rows), dtype=torch.uint8, device=dev)

    def check_input(self, image):
        if tuple(image.shape) != tuple(self.x.shape):
            raise AssertionError("Input size doesn't match model")

    def run(self, image, uniforms=None):
        self.check_input(image)
        with torch.cuda.device(self.eng.device):
            self.x.copy_(image, non_blocking=True)               # H2D from (pinned) host memory or D2D
            if self.uniforms is not None:
                self.uniforms.copy_(uniforms.to(torch.float32), non_blocking=True)
            if self.graph is None:
                self._launch()
            else:
                replay(self.eng.device, self.graph)
            return self._outputs()

    def _encode(self):
        eng = self.eng
        L.check(eng.lib.mdc_encode(eng.handle, L.ptr(self.x), self.B, None, L.ptr(self.memory), L.ptr(self.ws), self.ws_bytes,
                                   L.stream_ptr(eng.device)))

    def _reset_tokens(self):
        self.tokens.fill_(int(CFG.pad_idx))
        self.tokens[:, 0].fill_(int(CFG.bos_idx))

    def _init_prompt(self, width, prefill):
        """Prompted plans: the prompt (B, width) and its lengths are static buffers set before each run (set_prompt); with `prefill` = n
        the first n steps of every decoded row run as one all-positions pass (every row's prompt covers them)."""
        eng, dev = self.eng, self.eng.device
        self.prompt = self.prompt_len = self.prefill_ws = None
        self.prefill = int(prefill)
        if width:
            self.prompt = torch.full((self.B, width), int(CFG.pad_idx), dtype=torch.int32, device=dev)
            self.prompt_len = torch.zeros(self.B, dtype=torch.int32, device=dev)
        if self.prefill:
            rows = self.tokens.shape[0]
            self.prefill_ws = torch.empty(eng.lib.mdc_decode_prefill_workspace_bytes(eng.handle, rows, self.prefill), dtype=torch.uint8,
                                          device=dev)

    def set_prompt(self, prompt, lengths):
        """Host (or device) prompt int32 (B, prompt width), PAD past each row's length, and lengths int32 (B,), as check_prompt returns them."""
        with torch.cuda.device(self.eng.device):
            self.prompt.copy_(prompt, non_blocking=True)
            self.prompt_len.copy_(lengths, non_blocking=True)


class GenerationPlan(_Plan):
    """One (batch, new tokens, sampler, stop token) shape: encoder -> memory -> cross-K/V -> T decode steps.  With `use_graph` the
    whole call is one CUDA graph; with `split` it is two (encoder + cross-K/V | decode loop), `enc_graph` and `dec_graph`, so that a
    GenerationPipeline can run them on different streams.  `images_per_cluster` / `ctas_per_sm` override the decode launch options;
    the others come from decode_options."""

    def __init__(self, eng, B, T, top_k=0, top_p=1.0, want_logits=False, use_graph=True, split=False, eos_token=None,
                 images_per_cluster=None, ctas_per_sm=None, prompt_width=0, prefill=0):
        super().__init__(eng, B, T, B)
        d, dev = eng.dims, eng.device
        self.top_k, self.top_p, self.eos_token = int(top_k), float(top_p), eos_token
        self.images_per_cluster, self.ctas_per_sm = images_per_cluster, ctas_per_sm
        self.logits = torch.empty((B, T, d.vocab), dtype=torch.float32, device=dev) if want_logits else None
        if top_k != 0 or top_p != 1:
            self.uniforms = torch.zeros((B, T), dtype=torch.float32, device=dev)
        self._init_prompt(prompt_width, prefill)
        if split:
            self.enc_graph, self.dec_graph = capture_graphs(dev, self._launch_encode, self._launch_decode)
        elif use_graph:
            [self.graph] = capture_graphs(dev, self._launch)

    def _launch(self):
        self._launch_encode()
        self._launch_decode()

    def _launch_encode(self):
        eng = self.eng
        self._encode()
        L.check(eng.lib.mdc_cross_kv_build(eng.handle, L.ptr(self.memory), self.B, L.ptr(self.ckv), L.stream_ptr(eng.device)))

    def _launch_decode(self):
        self._reset_tokens()
        if self.prompt is not None:
            self.tokens[:, 1:1 + self.prompt.shape[1]].copy_(self.prompt)
        self.eng.decode(self.ckv, self.tokens, 0, self.T, max_tokens=self.T, forced=False, logits=self.logits, logits_row_offset=0,
                        confs=self.confs, uniforms=self.uniforms, top_k=self.top_k, top_p=self.top_p, kv=self.kv, scratch=self.scratch,
                        images_per_cluster=self.images_per_cluster, ctas_per_sm=self.ctas_per_sm, eos_token=self.eos_token,
                        prompt_len=self.prompt_len, prefill=self.prefill, prefill_ws=self.prefill_ws)

    def _outputs(self):
        return self.tokens, self.confs, self.logits


class BeamPlan(_Plan):
    """One beam-search shape (B images, T new tokens, K beams): encoder -> memory repeated K times -> cross-K/V of the B*K rows ->
    T x (teacher-forced decode step t, mdc_beam_step t) -> mdc_beam_finalize, captured as one CUDA graph with `use_graph`.
    The KV pool holds B*K rows of distinct pages (`own`, never rewritten); `kv.page_table` is the live table the decode kernels read,
    reset to `own` at the start of every run.  Prompted plans (`prompt_width` > 0) copy each image's prompt into all K of its token rows
    after the reset; with `prefill` = n, steps [0, n) of the B*K rows run as one all-positions pass (mdc_decode_prefill_steps) and the
    decode windows and beam steps start at t = n."""

    def __init__(self, eng, B, T, K, length_penalty, eos_token, use_graph, prompt_width=0, prefill=0):
        super().__init__(eng, B, T, B * K)
        d, dev, BK = eng.dims, eng.device, B * K
        self.K, self.length_penalty, self.eos_token = K, float(length_penalty), int(eos_token)
        self.memory_k = torch.empty((B, K, d.n_patches, d.dim), dtype=eng.dtype, device=dev)
        self.logits = torch.empty((BK, T, d.vocab), dtype=torch.float32, device=dev)
        self.own = self.kv.page_table.clone()
        self.scores = torch.empty(BK, dtype=torch.float32, device=dev)
        self.score0 = torch.full((B, K), -float("inf"), dtype=torch.float32, device=dev)
        self.score0[:, 0] = 0.0
        self.finish = torch.empty(BK, dtype=torch.int32, device=dev)
        self.lps = torch.zeros((BK, T), dtype=torch.float32, device=dev)
        self.beam_ws = torch.empty(eng.lib.mdc_beam_workspace_bytes(eng.handle, B, K), dtype=torch.uint8, device=dev)
        self.order = torch.empty((B, K), dtype=torch.int32, device=dev)
        self.norm = torch.empty((B, K), dtype=torch.float32, device=dev)
        self.rows = torch.arange(B, device=dev, dtype=torch.int64)[:, None] * K
        st = L.BeamState()
        st.B, st.K = B, K
        st.tokens, st.tokens_ld = self.tokens.data_ptr(), self.tokens.shape[1]
        st.kv_pool, st.page_table, st.own_pages = self.kv.pool.data_ptr(), self.kv.page_table.data_ptr(), self.own.data_ptr()
        st.pages_per_seq = self.kv.pages_per_seq
        st.scores, st.finish_step = self.scores.data_ptr(), self.finish.data_ptr()
        st.token_logprobs, st.token_logprobs_ld = self.lps.data_ptr(), T
        st.confs, st.confs_ld = self.confs.data_ptr(), self.confs.shape[1]
        st.eos_token = self.eos_token
        st.workspace, st.workspace_bytes = self.beam_ws.data_ptr(), self.beam_ws.numel()
        self._init_prompt(prompt_width, prefill)
        if self.prompt is not None:
            st.prompt_len = self.prompt_len.data_ptr()
        self.state = st
        if use_graph:
            [self.graph] = capture_graphs(dev, self._launch)

    def _launch(self):
        eng, B, K, T = self.eng, self.B, self.K, self.T
        d = eng.dims
        s = L.stream_ptr(eng.device)
        self._encode()
        self.memory_k.copy_(self.memory[:, None].expand_as(self.memory_k))
        L.check(eng.lib.mdc_cross_kv_build(eng.handle, L.ptr(self.memory_k), B * K, L.ptr(self.ckv), s))
        self._reset_tokens()
        if self.prompt is not None:
            P = self.prompt.shape[1]
            self.tokens.view(B, K, T + 1)[:, :, 1:1 + P].copy_(self.prompt[:, None].expand(B, K, P))
            self.lps.zero_()              # the prefill skips the beam steps t < n, which would otherwise write log-prob columns t
        self.kv.page_table.copy_(self.own)
        self.scores.copy_(self.score0.view(-1))
        self.finish.fill_(-1)
        if self.prefill:
            eng.decode(self.ckv, self.tokens, 0, self.prefill, max_tokens=T, forced=False, confs=self.confs, kv=self.kv,
                       scratch=self.scratch, prefill=self.prefill, prefill_ws=self.prefill_ws)
        row_bytes = d.vocab * self.logits.element_size()
        for t in range(self.prefill, T):
            eng.decode(self.ckv, self.tokens, t, t + 1, max_tokens=T, forced=True, logits=self.logits, logits_row_offset=0,
                       kv=self.kv, scratch=self.scratch)
            L.check(eng.lib.mdc_beam_step(eng.handle, C.byref(self.state), C.c_void_p(self.logits.data_ptr() + t * row_bytes),
                                          T * d.vocab, t, s))
        L.check(eng.lib.mdc_beam_finalize(eng.handle, C.byref(self.state), T, self.length_penalty, L.ptr(self.order),
                                          L.ptr(self.norm), s))

    def _outputs(self):
        rows = (self.rows + self.order.long()).view(-1)          # best-first gather of each image's rows
        B, K = self.B, self.K
        return (self.tokens[rows].view(B, K, -1), self.norm, self.lps[rows].view(B, K, -1), self.confs[rows].view(B, K, -1))
