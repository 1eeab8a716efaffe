"""mdc_model_create rejects decoder geometries the decode kernels do not cover (head width outside {32, 64, 128}, dim above 1024)
with a message that names the limit, before any kernel runs; Engine, built on a model's first call, reports the same error."""
import ctypes as C

import pytest
import torch

import mdcnet_b200 as M
from oracle import cases

L = M._lib

# (dim, heads, text the error names)
REJECTED = [
    (384, 8, "head width 48"),
    (1536, 12, "at most 1024"),
    (2048, 16, "at most 1024"),
]


def _dims(dim, heads):
    """A decoder-only geometry (no encoder blocks) with one decoder layer."""
    d = L.Dims()
    d.precision = L.MDC_BF16
    d.img_size, d.patch, d.in_chans = 16, 16, 3
    d.enc_dim, d.enc_depth, d.enc_heads, d.enc_mlp = 64, 0, 1, 256
    d.n_patches = 196
    d.dim, d.dec_heads, d.dec_layers, d.dec_ffn, d.vocab, d.max_pos = dim, heads, 1, 2048, 305, 99
    d.pad_idx, d.bos_idx, d.page_tokens = 302, 300, 16
    return d


def _model_create(d):
    """mdc_model_create with a table of NULL weights (the call only records the pointers); returns (rc, error text)."""
    lib = L.lib()
    n = lib.mdc_model_num_weights(C.byref(d))
    table = (C.c_void_p * n)()
    h = C.c_void_p()
    rc = lib.mdc_model_create(L.ctx("cuda:0"), C.byref(d), table, n, C.byref(h))
    if rc == 0:
        lib.mdc_model_destroy(h)
    return rc, lib.mdc_last_error().decode()


@pytest.mark.gpu
@pytest.mark.parametrize("dim,heads,names", REJECTED)
def test_model_create_rejects_uncovered_decoder(dim, heads, names):
    n0 = L.launch_count("cuda:0")
    rc, msg = _model_create(_dims(dim, heads))
    assert rc != 0
    assert names in msg, msg
    assert L.launch_count("cuda:0") == n0


@pytest.mark.gpu
def test_model_create_accepts_dim_1024_heads_8x128():
    rc, msg = _model_create(_dims(1024, 8))
    assert rc == 0, msg


@pytest.mark.gpu
@pytest.mark.parametrize("dim,heads,names", REJECTED)
def test_first_call_rejects_uncovered_decoder(dim, heads, names):
    Mc = cases.product_cfg(100)
    torch.manual_seed(0)
    enc = Mc.Encoder(model_name=cases.VIT, pretrained=False, out_dim=dim)
    model = Mc.EncoderDecoder(enc, Mc.Decoder(305, 196, dim, heads, 1)).eval().to("cuda:0")
    x = cases.images(2, seed=3).to("cuda:0")
    n0 = L.launch_count("cuda:0")
    with pytest.raises(L.MdcError, match=names):
        model.generate_tokens(x, 4)
    assert L.launch_count("cuda:0") == n0
