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
               images_per_cluster=None, ctas_per_sm=None, per_op_kernels=None, eos_token=None):
        """Runs decode steps [t_begin, t_end) back to back on the current stream (no host sync).  `eos_token` (free-running only): stop
        at that token -- after an image's first EOS its token columns are PAD and its confidences 0, and decoding ends once every image
        has finished (mdc_decode_state.stop_at_eos)."""
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
        with torch.cuda.device(self.device):
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
    @torch.no_grad()
    def generate_tokens(self, image, max_new_tokens, top_k=0, top_p=1.0, uniforms=None, return_logits=False, use_graph=None,
                        eos_token=None):
        """Returns (tokens int32 (B,1+T) on device, confs f32 (B,ceil(T/4)) on device[, logits (B,T,V)]).
        The whole call (encoder, cross-K/V, T decode steps) is one CUDA graph replay per (B, T, sampler, stop token) shape.
        `eos_token`: stop at that token (superset argument).  Up to and including an image's first EOS the result is bitwise the
        no-stop result; after it the tokens are PAD and the confidences 0, and decoding ends once every image has finished.  Not
        with `return_logits` (steps that do not run have no logits; predict()/forward() serve that use)."""
        eng = self._engine(image.device if image.is_cuda else None)
        d = eng.dims
        T = int(max_new_tokens)
        if T > d.max_pos:
            raise RuntimeError(f"max_len {T} exceeds CFG.max_len-1 = {d.max_pos}: the positional table has no more rows "
                               "(reference fails at model.py:93, Q6)")
        sampling = (top_k != 0 or top_p != 1)
        if eos_token is not None:
            if return_logits:
                raise ValueError("return_logits=True cannot be combined with eos_token: steps that do not run have no logits")
            eos_token = int(eos_token)
            if not 0 <= eos_token < d.vocab:
                raise ValueError(f"eos_token {eos_token} is outside the vocabulary [0, {d.vocab})")
        if use_graph is None:
            use_graph = os.environ.get("MDC_NO_GRAPH", "0") != "1"
        key = (id(eng), image.shape[0], T, int(top_k), float(top_p), bool(return_logits), bool(use_graph), eos_token, _decode_options_key())
        plans = self.__dict__.setdefault("_plans", {})
        if plans.get("eng") is not eng:
            plans.clear(); plans["eng"] = eng
        plan = plans.get(key)
        if plan is None:
            plan = GenerationPlan(eng, image.shape[0], T, top_k, top_p, sampling, return_logits, use_graph, eos_token=eos_token)
            plans[key] = plan
        if sampling and uniforms is None:
            uniforms = torch.rand((image.shape[0], T), dtype=torch.float32, device=eng.device)
        tokens, confs, logits = plan.run(image, uniforms)
        if return_logits:
            return tokens.clone(), confs.clone(), logits.clone()
        return tokens.clone(), confs.clone()

    @torch.no_grad()
    def generate_beam_tokens(self, image, max_new_tokens, num_beams, length_penalty=1.0, *, eos_token, use_graph=None):
        """Beam search (superset method; semantics in include/mdc_b200.h and DESIGN.md §3.4c).  Returns, on the device, each image's
        beams best first by length-normalised score: tokens int32 (B,K,1+T), normalised scores f32 (B,K), per-token log-probs f32
        (B,K,T) and confidences f32 (B,K,ceil(T/4)).  Tokens after a beam's EOS are PAD, with log-prob and confidence 0.  The whole
        call (encoder, cross-K/V for the B*K rows, T x (one teacher-forced decode step + one beam step), the final ordering) is one
        CUDA graph replay per (B, T, K, length penalty, stop token) shape."""
        eng = self._engine(image.device if image.is_cuda else None)
        d = eng.dims
        T, K = int(max_new_tokens), int(num_beams)
        if not 1 <= K <= 16:
            raise ValueError(f"num_beams {K} is outside 1..16")
        if not 1 <= T <= d.max_pos:
            raise RuntimeError(f"max_len {T} is outside 1..CFG.max_len-1 = {d.max_pos}: the positional table has no more rows "
                               "(reference fails at model.py:93, Q6)")
        eos_token = int(eos_token)
        if not 0 <= eos_token < d.vocab:
            raise ValueError(f"eos_token {eos_token} is outside the vocabulary [0, {d.vocab})")
        if use_graph is None:
            use_graph = os.environ.get("MDC_NO_GRAPH", "0") != "1"
        key = ("beam", id(eng), image.shape[0], T, K, float(length_penalty), eos_token, bool(use_graph), _decode_options_key())
        plans = self.__dict__.setdefault("_plans", {})
        if plans.get("eng") is not eng:
            plans.clear(); plans["eng"] = eng
        plan = plans.get(key)
        if plan is None:
            plan = BeamPlan(eng, image.shape[0], T, K, float(length_penalty), eos_token, use_graph)
            plans[key] = plan
        return tuple(o.clone() for o in plan.run(image))


class GenerationPlan:
    """Static buffers + (optionally) a captured CUDA graph for one (batch, new tokens, sampler) shape:
    encoder -> memory -> cross-K/V -> T decode steps, no host synchronisation anywhere inside."""

    def __init__(self, eng, B, T, top_k, top_p, sampling, want_logits, use_graph, split=False, images_per_cluster=None, ctas_per_sm=None,
                 eos_token=None):
        # everything below (allocations, warm-up launches, graph capture) on the ENGINE's device: torch.cuda.graph captures the current
        # device's stream, so with another device current the capture came back empty and replays did nothing (two-device test)
        with torch.cuda.device(eng.device):
            self._build(eng, B, T, top_k, top_p, sampling, want_logits, use_graph, split, images_per_cluster, ctas_per_sm, eos_token)

    def _build(self, eng, B, T, top_k, top_p, sampling, want_logits, use_graph, split, images_per_cluster, ctas_per_sm, eos_token):
        d = eng.dims
        dev = eng.device
        self.eng, self.B, self.T = eng, B, T
        self.top_k, self.top_p = int(top_k), float(top_p)
        self.eos_token = eos_token
        self.images_per_cluster = _DECODE_OPTIONS["images_per_cluster"] if images_per_cluster is None else int(images_per_cluster)
        self.ctas_per_sm = _DECODE_OPTIONS["ctas_per_sm"] if ctas_per_sm is None else int(ctas_per_sm)
        self.per_op_kernels = bool(_DECODE_OPTIONS["per_op_kernels"])
        self.x = torch.zeros((B, d.in_chans, d.img_size, d.img_size), dtype=torch.float32, device=dev)
        self.ws_bytes = eng.lib.mdc_encode_workspace_bytes(eng.handle, B)
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.memory = torch.empty((B, d.n_patches, d.dim), dtype=eng.dtype, device=dev)
        self.ckv = torch.empty(eng.lib.mdc_cross_kv_bytes(eng.handle, B), dtype=torch.uint8, device=dev)
        self.tokens = torch.empty((B, T + 1), dtype=torch.int32, device=dev)
        self.confs = torch.zeros((B, (T + 3) // 4), dtype=torch.float32, device=dev)
        self.logits = torch.empty((B, T, d.vocab), dtype=torch.float32, device=dev) if want_logits else None
        self.uniforms = torch.zeros((B, T), dtype=torch.float32, device=dev) if sampling else None
        self.kv = PagedKVCache(B, T, d.dec_layers, d.dim, d.page_tokens, eng.dtype, dev)
        self.scratch = torch.empty(eng.lib.mdc_decode_workspace_bytes(eng.handle, B), dtype=torch.uint8, device=dev)
        self.graph = None
        self.split = bool(split)
        if split:
            # two graphs (encoder + cross-K/V | decode loop) so that a GenerationPipeline can run them on different streams
            assert use_graph, "split plans are graph plans"
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                self._launch_encode(); self._launch_decode()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            self.enc_graph, self.dec_graph = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            n0 = L.launch_count(dev)
            with torch.cuda.graph(self.enc_graph, stream=side):     # an explicit capture stream of THIS device (torch's default one is a
                                                                    # process-wide singleton on whichever device captured first)
                self._launch_encode()
            n1 = L.launch_count(dev)
            with torch.cuda.graph(self.dec_graph, stream=side):
                self._launch_decode()
            self.enc_kernels, self.dec_kernels = n1 - n0, L.launch_count(dev) - n1
            self.enc_done, self.dec_done = torch.cuda.Event(), torch.cuda.Event()
            self.busy = False
            return
        if use_graph:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                self._launch()                      # warm-up: tensor maps, smem attributes, lazy module load
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            n0 = L.launch_count(dev)
            with torch.cuda.graph(g, stream=side):
                self._launch()
            self.graph_kernels = L.launch_count(dev) - n0      # kernels of libmdc_b200.so inside one replay
            self.graph = g

    def _launch(self):
        self._launch_encode()
        self._launch_decode()

    def _launch_encode(self):
        eng = self.eng
        with torch.cuda.device(eng.device):
            L.check(eng.lib.mdc_encode(eng.handle, L.ptr(self.x), self.B, None, L.ptr(self.memory), L.ptr(self.ws), self.ws_bytes, L.stream_ptr(eng.device)))
            L.check(eng.lib.mdc_cross_kv_build(eng.handle, L.ptr(self.memory), self.B, L.ptr(self.ckv), L.stream_ptr(eng.device)))

    def _launch_decode(self):
        eng = self.eng
        self.tokens.fill_(int(CFG.pad_idx))
        self.tokens[:, 0].fill_(int(CFG.bos_idx))
        eng.decode(self.ckv, self.tokens, 0, self.T, max_tokens=self.T, forced=False, logits=self.logits, logits_row_offset=0,
                   confs=self.confs, uniforms=self.uniforms, top_k=self.top_k, top_p=self.top_p, kv=self.kv, scratch=self.scratch,
                   images_per_cluster=self.images_per_cluster, ctas_per_sm=self.ctas_per_sm, per_op_kernels=self.per_op_kernels,
                   eos_token=self.eos_token)

    def run(self, image, uniforms=None):
        d = self.eng.dims
        if tuple(image.shape) != tuple(self.x.shape):
            raise AssertionError("Input size doesn't match model")
        with torch.cuda.device(self.eng.device):
            self.x.copy_(image, non_blocking=True)               # H2D from (pinned) host memory or D2D
            if self.uniforms is not None:
                self.uniforms.copy_(uniforms.to(torch.float32), non_blocking=True)
            if self.graph is not None:
                self.graph.replay()
                L.note_graph_replay(self.eng.device, self.graph_kernels)
            else:
                self._launch()
        return self.tokens, self.confs, self.logits


class BeamPlan:
    """Static buffers + (optionally) a captured CUDA graph for one beam-search shape (B images, T new tokens, K beams): encoder ->
    memory repeated K times -> cross-K/V of the B*K rows -> T x (teacher-forced decode step t, mdc_beam_step t) -> mdc_beam_finalize.
    The KV pool holds B*K rows of distinct pages (`own`, never rewritten); `kv.page_table` is the live table the decode kernels read,
    reset to `own` at the start of every run."""

    def __init__(self, eng, B, T, K, length_penalty, eos_token, use_graph):
        with torch.cuda.device(eng.device):
            self._build(eng, B, T, K, length_penalty, eos_token, use_graph)

    def _build(self, eng, B, T, K, length_penalty, eos_token, use_graph):
        d = eng.dims
        dev = eng.device
        BK = B * K
        self.eng, self.B, self.T, self.K = eng, B, T, K
        self.length_penalty, self.eos_token = float(length_penalty), int(eos_token)
        self.x = torch.zeros((B, d.in_chans, d.img_size, d.img_size), dtype=torch.float32, device=dev)
        self.ws_bytes = eng.lib.mdc_encode_workspace_bytes(eng.handle, B)
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.memory = torch.empty((B, d.n_patches, d.dim), dtype=eng.dtype, device=dev)
        self.memory_k = torch.empty((B, K, d.n_patches, d.dim), dtype=eng.dtype, device=dev)
        self.ckv = torch.empty(eng.lib.mdc_cross_kv_bytes(eng.handle, BK), dtype=torch.uint8, device=dev)
        self.tokens = torch.empty((BK, T + 1), dtype=torch.int32, device=dev)
        self.logits = torch.empty((BK, T, d.vocab), dtype=torch.float32, device=dev)
        self.kv = PagedKVCache(BK, T, d.dec_layers, d.dim, d.page_tokens, eng.dtype, dev)
        self.own = self.kv.page_table.clone()
        self.scratch = torch.empty(eng.lib.mdc_decode_workspace_bytes(eng.handle, BK), dtype=torch.uint8, device=dev)
        self.scores = torch.empty(BK, dtype=torch.float32, device=dev)
        self.score0 = torch.full((B, K), -float("inf"), dtype=torch.float32, device=dev)
        self.score0[:, 0] = 0.0
        self.finish = torch.empty(BK, dtype=torch.int32, device=dev)
        self.lps = torch.zeros((BK, T), dtype=torch.float32, device=dev)
        self.confs = torch.zeros((BK, (T + 3) // 4), dtype=torch.float32, device=dev)
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
        self.state = st
        self.graph = None
        if use_graph:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                self._launch()                      # warm-up: tensor maps, smem attributes, lazy module load
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            n0 = L.launch_count(dev)
            with torch.cuda.graph(g, stream=side):
                self._launch()
            self.graph_kernels = L.launch_count(dev) - n0
            self.graph = g

    def _launch(self):
        eng, B, K, T = self.eng, self.B, self.K, self.T
        d = eng.dims
        s = L.stream_ptr(eng.device)
        with torch.cuda.device(eng.device):
            L.check(eng.lib.mdc_encode(eng.handle, L.ptr(self.x), B, None, L.ptr(self.memory), L.ptr(self.ws), self.ws_bytes, s))
            self.memory_k.copy_(self.memory[:, None].expand_as(self.memory_k))
            L.check(eng.lib.mdc_cross_kv_build(eng.handle, L.ptr(self.memory_k), B * K, L.ptr(self.ckv), s))
            self.tokens.fill_(int(CFG.pad_idx))
            self.tokens[:, 0].fill_(int(CFG.bos_idx))
            self.kv.page_table.copy_(self.own)
            self.scores.copy_(self.score0.view(-1))
            self.finish.fill_(-1)
            row_bytes = d.vocab * self.logits.element_size()
            for t in range(T):
                eng.decode(self.ckv, self.tokens, t, t + 1, max_tokens=T, forced=True, logits=self.logits, logits_row_offset=0,
                           kv=self.kv, scratch=self.scratch)
                L.check(eng.lib.mdc_beam_step(eng.handle, C.byref(self.state), C.c_void_p(self.logits.data_ptr() + t * row_bytes),
                                              T * d.vocab, t, s))
            L.check(eng.lib.mdc_beam_finalize(eng.handle, C.byref(self.state), T, self.length_penalty, L.ptr(self.order),
                                              L.ptr(self.norm), s))

    def run(self, image):
        if tuple(image.shape) != tuple(self.x.shape):
            raise AssertionError("Input size doesn't match model")
        with torch.cuda.device(self.eng.device):
            self.x.copy_(image, non_blocking=True)
            if self.graph is not None:
                self.graph.replay()
                L.note_graph_replay(self.eng.device, self.graph_kernels)
            else:
                self._launch()
            rows = (self.rows + self.order.long()).view(-1)          # best-first gather of each image's rows
            B, K = self.B, self.K
            return (self.tokens[rows].view(B, K, -1), self.norm, self.lps[rows].view(B, K, -1), self.confs[rows].view(B, K, -1))
