"""Thin helpers for the GPU tests: call the C ABI directly (raw pointers + current stream)."""
import torch

import mdcnet_b200 as M

L = M._lib


def dtype_code(dtype):
    """The library's element-type code, including IEEE half (mdc_gemm's fp16 mode)."""
    return L.MDC_F16 if dtype == torch.float16 else L.dtype_code(dtype)


def gemm(A, W, dtype, epilogue, bias=None, aux0=None, period=0, R=None, D=None):
    """Calls mdc_gemm.  A [M,K], W [N,K] in `dtype` (row strides taken from the tensors, so column / row slices pass as
    they are); returns D (or the updated f32 stream R).  `D`: an output view to write into instead of a new tensor."""
    dev = A.device
    Mr, K = A.shape
    N = W.shape[0]
    code = dtype_code(dtype)
    if epilogue in (L.EPI_LS_RESIDUAL, L.EPI_PATCH):
        D = R
    elif D is None:
        D = torch.empty((Mr, N), dtype=dtype, device=dev)
    L.check(L.lib().mdc_gemm(L.ctx(dev), code, epilogue, L.ptr(A), A.stride(0), L.ptr(W), W.stride(0), L.ptr(D), D.stride(0),
                             L.ptr(bias), L.ptr(aux0), period, Mr, N, K, L.stream_ptr()))
    return D


def strip_attention(qkv, n_strips, strip_len, heads, hd, scale, soq=0, out=None):
    """`out`: an output view (any row stride) to write into instead of a new tensor."""
    if out is None:
        out = torch.empty((qkv.shape[0], heads * hd), dtype=qkv.dtype, device=qkv.device)
    L.check(L.lib().mdc_strip_attention(L.ctx(qkv.device), L.dtype_code(qkv.dtype), L.ptr(qkv), qkv.stride(0), L.ptr(out), out.stride(0),
                                        n_strips, strip_len, heads, hd, float(scale), soq, L.stream_ptr()))
    return out


def layernorm(x, w, b, eps, out_dtype, out=None):
    """`out`: an output view (any row stride) to write into instead of a new tensor."""
    if out is None:
        out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    L.check(L.lib().mdc_layernorm(L.ctx(x.device), L.ptr(x), x.stride(0), L.ptr(w), L.ptr(b), eps, L.ptr(out), out.stride(0),
                                  L.dtype_code(out_dtype), x.shape[0], x.shape[1], L.stream_ptr()))
    return out


def select(logits, top_k=0, top_p=1.0, uniforms=None):
    B, V = logits.shape
    tok = torch.empty(B, dtype=torch.int32, device=logits.device)
    conf = torch.empty(B, dtype=torch.float32, device=logits.device)
    L.check(L.lib().mdc_select(L.ctx(logits.device), L.ptr(logits), logits.stride(0), B, V, top_k, float(top_p), L.ptr(uniforms),
                               L.ptr(tok), L.ptr(conf), None, L.stream_ptr()))
    return tok, conf


def cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return (a @ b / (a.norm() * b.norm())).item()
