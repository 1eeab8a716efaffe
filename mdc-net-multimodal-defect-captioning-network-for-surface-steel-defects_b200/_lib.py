"""ctypes binding of libmdc_b200.so (the C ABI declared in include/mdc_b200.h).

The product path has NO CPU fallback: `lib()` raises if the shared library is missing, and
`ctx(device)` raises if there is no sm_100 CUDA device.  Every call passes raw device pointers
(`tensor.data_ptr()`) plus the current torch CUDA stream, so the work is ordered with torch's
allocator/streams and can be captured into a CUDA graph.
"""
import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MDC_LIB_PATH") or os.path.join(_HERE, "libmdc_b200.so")     # env override: A/B runs of two builds (tools/)

MDC_F32, MDC_BF16, MDC_F16 = 0, 1, 2
EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_RELU, EPI_LS_RESIDUAL, EPI_PATCH = range(5)
IOU_EPS, IOU_PLAIN, IOU_NAN0, IOU_GIOU = range(4)

# slot enums (must match include/mdc_b200.h)
ENC_GLOBAL = ["W_PATCH", "B_PATCH", "CLS", "POS", "NORM_W", "NORM_B"]
ENC_BLOCK = ["N1_W", "N1_B", "QKV_W", "QKV_B", "PROJ_W", "PROJ_B", "LS1",
             "N2_W", "N2_B", "FC1_W", "FC1_B", "FC2_W", "FC2_B", "LS2"]
DEC_GLOBAL = ["EMB", "DEC_POS", "ENC_POS", "OUT_W", "OUT_B", "AX_QKV_W", "AX_OUT_W", "AX_OUT_B"]
DEC_LAYER = ["SA_IN_W", "SA_IN_B", "SA_OUT_W", "SA_OUT_B", "LN1_W", "LN1_B",
             "CA_IN_W", "CA_IN_B", "CA_OUT_W", "CA_OUT_B", "LN2_W", "LN2_B",
             "FF1_W", "FF1_B", "FF2_W", "FF2_B", "LN3_W", "LN3_B"]


class Dims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "precision", "img_size", "patch", "in_chans", "enc_dim", "enc_depth", "enc_heads", "enc_mlp",
        "n_patches", "dim", "dec_heads", "dec_layers", "dec_ffn", "vocab", "max_pos", "pad_idx", "bos_idx",
        "has_axial", "page_tokens")]


class TokenGrammar(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("pad", "eos", "caption_start", "caption_end", "label_lo", "label_hi", "coord_max",
                                         "num_bins", "width", "height")]


TOK_BBOXES, TOK_DECODE = 0, 1


class DecodeState(C.Structure):
    _fields_ = [
        ("B", C.c_int32),
        ("tokens", C.c_void_p), ("tokens_ld", C.c_int32),
        ("kv_pool", C.c_void_p), ("page_table", C.c_void_p), ("pages_per_seq", C.c_int32), ("n_pages", C.c_int32),
        ("cross_kv", C.c_void_p),
        ("logits", C.c_void_p), ("logits_ld", C.c_int32), ("logits_row_offset", C.c_int32),
        ("confs", C.c_void_p), ("confs_ld", C.c_int32),
        ("uniforms", C.c_void_p), ("uniforms_ld", C.c_int32),
        ("top_k", C.c_int32), ("top_p", C.c_float),
        ("forced", C.c_int32),
        ("pos_override", C.c_void_p),
        ("x_override", C.c_void_p), ("x_override_ld", C.c_int32),
        ("scratch", C.c_void_p), ("scratch_bytes", C.c_size_t),
        ("images_per_cluster", C.c_int32),
        ("ctas_per_sm", C.c_int32),
        ("per_op_kernels", C.c_int32),
        ("stop_at_eos", C.c_int32), ("eos_token", C.c_int32),
    ]


class BeamState(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("K", C.c_int32),
        ("tokens", C.c_void_p), ("tokens_ld", C.c_int32),
        ("kv_pool", C.c_void_p), ("page_table", C.c_void_p), ("own_pages", C.c_void_p), ("pages_per_seq", C.c_int32),
        ("scores", C.c_void_p), ("finish_step", C.c_void_p),
        ("token_logprobs", C.c_void_p), ("token_logprobs_ld", C.c_int32),
        ("confs", C.c_void_p), ("confs_ld", C.c_int32),
        ("eos_token", C.c_int32),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
    ]


_P, _I, _L, _F, _SZ = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); the complete export list of include/mdc_b200.h
SIGNATURES = {
    "mdc_abi_version": (_I, []),
    "mdc_last_error": (C.c_char_p, []),
    "mdc_ctx_create": (_I, [_I, C.POINTER(_P)]),
    "mdc_ctx_destroy": (_I, [_P]),
    "mdc_ctx_launch_count": (_L, [_P]),
    "mdc_gemm": (_I, [_P, _I, _I, _P, _L, _P, _L, _P, _L, _P, _P, _I, _I, _I, _I, _P]),
    "mdc_strip_attention": (_I, [_P, _I, _P, _L, _P, _L, _I, _I, _I, _I, _F, _I, _P]),
    "mdc_layernorm": (_I, [_P, _P, _L, _P, _P, _F, _P, _L, _I, _I, _I, _P]),
    "mdc_preprocess_gray": (_I, [_P, _P, _I, _I, _I, _P, _I, _P]),
    "mdc_preprocess_bgr": (_I, [_P, _P, _I, _I, _I, _P, _I, _P]),
    "mdc_interp_rows": (_I, [_P, _P, _I, _P, _I, _I, _P]),
    "mdc_model_create": (_I, [_P, C.POINTER(Dims), C.POINTER(_P), _I, C.POINTER(_P)]),
    "mdc_model_destroy": (_I, [_P]),
    "mdc_model_num_weights": (_I, [C.POINTER(Dims)]),
    "mdc_encode_workspace_bytes": (_SZ, [_P, _I]),
    "mdc_encode": (_I, [_P, _P, _I, _P, _P, _P, _SZ, _P]),
    "mdc_memory_from_encoder_out": (_I, [_P, _P, _I, _P, _P]),
    "mdc_cross_kv_bytes": (_SZ, [_P, _I]),
    "mdc_cross_kv_build": (_I, [_P, _P, _I, _P, _P]),
    "mdc_decode_workspace_bytes": (_SZ, [_P, _I]),
    "mdc_decode_pack_bytes": (_SZ, [_P]),
    "mdc_decode_pack": (_I, [_P, _P, _P]),
    "mdc_kv_page_bytes": (_SZ, [_P]),
    "mdc_decode_steps": (_I, [_P, C.POINTER(DecodeState), _I, _I, _P]),
    "mdc_decoder_prefill_workspace_bytes": (_SZ, [_P, _I, _I]),
    "mdc_decoder_prefill": (_I, [_P, _P, _I, _I, _I, _P, _P, _P, _I, _I, _I, _P, _SZ, _P]),
    "mdc_beam_workspace_bytes": (_SZ, [_P, _I, _I]),
    "mdc_beam_step": (_I, [_P, C.POINTER(BeamState), _P, _L, _I, _P]),
    "mdc_beam_finalize": (_I, [_P, C.POINTER(BeamState), _I, _F, _P, _P, _P]),
    "mdc_select": (_I, [_P, _P, _L, _I, _I, _I, _F, _P, _P, _P, _P, _P]),
    "mdc_axial_workspace_bytes": (_SZ, [_P, _I, _I]),
    "mdc_axial_attention": (_I, [_P, _P, _I, _I, _I, _P, _P, _SZ, _P]),
    "mdc_axial_embed_workspace_bytes": (_SZ, [_P, _I, _I]),
    "mdc_axial_embed": (_I, [_P, _P, _I, _I, _I, _P, _I, _P, _P, _SZ, _P]),
    "mdc_iou_batch": (_I, [_P, _I, _P, _P, _I, _I, _I, _P, _P, _P]),
    "mdc_giou_loss": (_I, [_P, _P, _P, _I, _I, _I, _F, _P, _P, _P, _P]),
    "mdc_map_match": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _I, _P, _P, _P]),
    "mdc_decode_tokens": (_I, [_P, _I, _P, _L, _I, _I, C.POINTER(TokenGrammar), _I, _P, _P, _P, _P, _P, _P]),
}

_lib = None
_ctxs = {}
_lock = threading.Lock()


class MdcError(RuntimeError):
    pass


def lib():
    """Load the shared library (building nothing: run __graft_entry__.build() / build.py first)."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise MdcError(f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build`; "
                                   "this package has no CPU / PyTorch fallback")
                l = C.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(l, name)
                    fn.restype, fn.argtypes = res, args
                _lib = l
    return _lib


def check(rc):
    if rc != 0:
        raise MdcError(f"libmdc_b200: error {rc}: {lib().mdc_last_error().decode()}")


def ctx(device=None):
    """One mdc_ctx per CUDA device index."""
    if not torch.cuda.is_available():
        raise MdcError("no CUDA device: the MDC-Net B200 path has no CPU fallback")
    idx = torch.cuda.current_device() if device is None else torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    if idx not in _ctxs:
        with _lock:
            if idx not in _ctxs:
                h = _P()
                check(lib().mdc_ctx_create(idx, C.byref(h)))
                _ctxs[idx] = h
    return _ctxs[idx]


_replayed = {}


def _dev_index(device=None):
    idx = torch.cuda.current_device() if device is None else torch.device(device).index
    return torch.cuda.current_device() if idx is None else idx


def note_graph_replay(device, n_kernels):
    """A CUDA-graph replay re-launches the `n_kernels` kernels counted while the graph was captured; the C side only
    sees the capture, so replays are accounted here."""
    i = _dev_index(device)
    _replayed[i] = _replayed.get(i, 0) + int(n_kernels)


def launch_count(device=None):
    """Kernels of libmdc_b200.so launched on `device` so far: direct launches (counted in C, mdc_ctx_launch_count)
    plus the kernels inside replayed CUDA graphs."""
    return int(lib().mdc_ctx_launch_count(ctx(device))) + _replayed.get(_dev_index(device), 0)


def stream_ptr(device=None):
    """The current torch stream of `device` (default: the current device)."""
    return _P(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  The tensor must be contiguous where the ABI says so."""
    if t is None:
        return _P(0)
    return _P(t.data_ptr())


def dtype_code(dt):
    if dt == torch.float32:
        return MDC_F32
    if dt == torch.bfloat16:
        return MDC_BF16
    raise MdcError(f"unsupported dtype {dt}")
