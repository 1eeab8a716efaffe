"""GPU: every kernel instantiation the encoder-side dispatchers (mdc_gemm, mdc_strip_attention, mdc_layernorm) select on a
148-SM B200, against float64 computed on the GPU from the same rounded operands the kernel sees; strided operands with the
memory around them left bit-for-bit untouched; fp16 saturation; and the argument checks that reject misaligned operands
before any launch.

GEMM bound, per element (u = 2^-24):
    (K + 1) * u * (|A| @ |W|^T + |bias|)     K fp32 accumulation steps and the bias add
scaled by the epilogue's Lipschitz constant (|GELU'| <= 1.13, plus the 3e-7 error of the epilogue's GELU polynomial; |gamma|
for LayerScale), plus the rounding of the output: 2^-8 |want| for bf16, 2^-11 |want| for fp16, 2u |want| for the f32 stream
(LayerScale product and residual add).  A dropped K block, a bias or gamma from the wrong column or a wrong row in the second
CTA of a pair errs by orders of magnitude more than this."""
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

import mdcnet_b200 as M  # noqa: E402
from oracle import cases, mdc_oracle as O  # noqa: E402
from tests import gpu_util as G  # noqa: E402

L = M._lib
DEV = "cuda"
U = 2.0 ** -24
OUT_RND = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11, torch.float32: 2 * U}
GELU_LIP, GELU_ERR = 1.13, 3e-7
BIAS, GELU, RELU, LS, PATCH = L.EPI_BIAS, L.EPI_BIAS_GELU, L.EPI_BIAS_RELU, L.EPI_LS_RESIDUAL, L.EPI_PATCH
EPI_NAME = {BIAS: "bias", GELU: "gelu", RELU: "relu", LS: "ls_residual", PATCH: "patch"}

# (M, N, K, epilogue, period) and the tile gemm_tc_launch selects on 148 SMs: BN = 256 when N % 256 == 0 and 128 x 256 tiles give
# every SM one; BN = 64 when 128 x 128 tiles would not; else BN = 128.  CTA pairs for BN >= 128 and M >= 256, except PATCH.
GEMM_CASES = [
    # BN = 64, one CTA: 4 x 5 tiles; K = 200 and 72 end in a partial 64-wide K block (TMA zero fill), N = 520 in an 8-column tail
    *[(394, 520, 200, e, 0) for e in (BIAS, GELU, RELU, LS)],
    (392, 512, 72, PATCH, 196),
    # BN = 128, one CTA: M < 256, 2 x 75 tiles of 128 columns (N % 256 = 8)
    *[(200, 9480, 64, e, 0) for e in (BIAS, GELU, RELU, LS)],
    (4704, 512, 768, PATCH, 196),                    # patch embedding at B = 24: 37 x 4 tiles
    # BN = 256, one CTA: 2 x 74 tiles of 256 columns
    *[(200, 18944, 64, e, 0) for e in (BIAS, GELU, RELU, LS)],
    (12544, 512, 768, PATCH, 196),                   # patch embedding at B = 64: 98 x 2 tiles; 32-row chunks cross images
    # BN = 128, CTA pairs: 16 x 12 tiles
    (2000, 1536, 512, GELU, 0), (2000, 1536, 512, LS, 0),
    # BN = 128, CTA pairs: the second CTA of the last row pair (rows 4224..) has no valid row; 8-column N tail
    *[(4196, 1544, 512, e, 0) for e in (BIAS, RELU, LS)],
    # BN = 256, CTA pairs: 19 x 8 tiles; the last pair has 96 valid rows, all in its first CTA
    *[(2400, 2048, 128, e, 0) for e in (BIAS, GELU, RELU, LS)],
]
# fp16 mode (the decoder prefill): BN = 64 (4 x 12 tiles), 128 (16 x 12), 256 (50 x 3 and 50 x 4); bias / bias + ReLU only
F16_CASES = [(s, e) for s in ((394, 768, 256), (2000, 1536, 256), (6336, 768, 256), (6336, 1024, 256)) for e in (BIAS, RELU)]


def _randn(shape, seed, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(DEV)


def _case_id(c):
    return f"{c[0]}x{c[1]}x{c[2]}-{EPI_NAME[c[3]]}"


def _gemm_ref(A, W, bias, epi, gamma=None, R0=None, pos=None, period=0):
    """fp64 result of the epilogue on the whole output (R for LS_RESIDUAL / PATCH) and its bound before output rounding."""
    a, w = A.double(), W.double()
    K = a.shape[1]
    acc, mag = a @ w.T, a.abs() @ w.abs().T
    if bias is not None:
        acc, mag = acc + bias.double(), mag + bias.double().abs()
    err = (K + 1) * U * mag
    if epi == BIAS:
        return acc, err
    if epi == GELU:
        return torch.nn.functional.gelu(acc), GELU_LIP * err + GELU_ERR
    if epi == RELU:
        return torch.relu(acc), err
    if epi == LS:
        return R0.double() + gamma.double() * acc, gamma.double().abs() * err
    # PATCH: row r of the product lands on row r + r // period + 1 of R (each image's cls row is skipped), plus pos[r % period]
    r = torch.arange(acc.shape[0], device=DEV)
    dst = r + r // period + 1
    want, bound = R0.double().clone(), torch.zeros_like(R0, dtype=torch.float64)
    want[dst] = acc + pos.double()[r % period]
    bound[dst] = err
    return want, bound


def _assert_within(got, want, err, out_dtype, what):
    bound = err + OUT_RND[out_dtype] * want.abs()
    d = (got.double() - want).abs()
    bad = d > bound
    assert not bad.any(), (what, f"{int(bad.sum())} elements out of bound, first at {bad.nonzero()[0].tolist()}",
                           f"max |d| / bound = {(d / bound.clamp_min(1e-30)).max().item():.3g}")


def _gemm_operands(case, dtype):
    Mr, N, K, epi, period = case
    A, W = _randn((Mr, K), 1, 0.5).to(dtype), _randn((N, K), 2, 0.5).to(dtype)
    bias, aux0, R0 = _randn((N,), 3), None, None
    if epi == LS:
        aux0, R0 = _randn((N,), 4), _randn((Mr, N), 5)
    elif epi == PATCH:
        aux0, R0 = _randn((period, N), 6), torch.full((Mr + Mr // period, N), 7.0, device=DEV)
    return A, W, bias, aux0, R0


@pytest.mark.parametrize("case", GEMM_CASES, ids=_case_id)
def test_gemm_instantiation_against_fp64(case):
    """The same bf16-rounded operands through the tensor-core kernel (bf16) and the FFMA kernel (fp32), both against fp64."""
    Mr, N, K, epi, period = case
    A, W, bias, aux0, R0 = _gemm_operands(case, torch.bfloat16)
    want, err = _gemm_ref(A, W, bias, epi, gamma=aux0, R0=R0, pos=aux0, period=period)
    for dt in (torch.bfloat16, torch.float32):
        R = None if R0 is None else R0.clone()
        got = G.gemm(A.to(dt), W.to(dt), dt, epi, bias=bias, aux0=aux0, period=period, R=R)
        _assert_within(got, want, err, torch.float32 if R0 is not None else dt, (case, dt))


@pytest.mark.parametrize("case", F16_CASES, ids=lambda c: f"{c[0][0]}x{c[0][1]}x{c[0][2]}-{EPI_NAME[c[1]]}")
def test_gemm_fp16_mode_against_fp64(case):
    (Mr, N, K), epi = case
    A, W = _randn((Mr, K), 1, 0.5).half(), _randn((N, K), 2, 0.5).half()
    bias = _randn((N,), 3)
    want, err = _gemm_ref(A, W, bias, epi)
    _assert_within(G.gemm(A, W, torch.float16, epi, bias=bias), want, err, torch.float16, (case, "fp16"))
    _assert_within(G.gemm(A.float(), W.float(), torch.float32, epi, bias=bias), want, err, torch.float32, (case, "fp32"))


def test_gemm_fp16_saturates_to_the_finite_range():
    """acc + bias reaches +-1e5 in some columns: those outputs are exactly +-65504 (never inf); every other output is the fp16
    rounding of the fp64 value (one fp16 ulp plus the accumulation bound).  GELU, LayerScale and PATCH have no fp16 form."""
    Mr, N, K = 394, 768, 256
    A, W = _randn((Mr, K), 1, 0.5).half(), _randn((N, K), 2, 0.5).half()
    bias = _randn((N,), 3)
    bias[0::8], bias[3::8] = 1e5, -1e5
    for epi in (BIAS, RELU):
        want, err = _gemm_ref(A, W, bias, epi)
        got = G.gemm(A, W, torch.float16, epi, bias=bias).double()
        sat = want.abs() > 65504
        assert sat[:, 0::8].all() and (epi == RELU or sat[:, 3::8].all())
        assert torch.equal(got[sat], want[sat].sign() * 65504), EPI_NAME[epi]
        ok = ~sat
        ulp = torch.exp2(torch.floor(torch.log2(want[ok].abs().clamp_min(2.0 ** -14))) - 10)
        d = (got[ok] - want[ok]).abs()
        assert (d <= ulp + err[ok]).all(), (EPI_NAME[epi], (d / (ulp + err[ok])).max().item())
    A16 = A[:256]
    for epi in (GELU, LS, PATCH):
        R = torch.zeros((264, N), device=DEV)
        with pytest.raises(L.MdcError):
            G.gemm(A16, W, torch.float16, epi, bias=bias, aux0=torch.zeros((256, N), device=DEV), period=128, R=R)


@pytest.mark.parametrize("dtype,K", [(torch.bfloat16, 72), (torch.bfloat16, 200), (torch.float32, 20), (torch.float32, 36)])
def test_gemm_strided_operands_leave_the_rest_untouched(dtype, K):
    """A is a column slice (lda = K + 64), W a row slice at offset K*K (as the cross-K/V build passes the in-projection), D the
    columns [16, 16 + N) of a buffer with ldd = N + 32 and rows to spare; the PATCH table has the same stride ldd.  Every byte
    outside the written block keeps its sentinel; bias = NULL is honoured on both kernels."""
    Mr, N, period = 300, 136, 100
    Abuf = _randn((Mr, K + 64), 1, 0.5).to(dtype)
    A = Abuf[:, :K]
    Wbuf = _randn((K + N, K), 2, 0.5).to(dtype)
    W = Wbuf[K:]
    bias, gamma = _randn((N,), 3), _randn((N,), 4)
    ldd = N + 32

    def window(buf, rows):
        return buf[:rows, 16:16 + N]

    def untouched(buf, rows, sentinel):
        outside = torch.ones_like(buf, dtype=torch.bool)
        outside[:rows, 16:16 + N] = False
        return torch.equal(buf[outside], sentinel[outside])

    for b in (bias, None):
        Dbuf = torch.full((Mr + 3, ldd), -3.0, dtype=dtype, device=DEV)
        G.gemm(A, W, dtype, BIAS, bias=b, D=window(Dbuf, Mr))
        want, err = _gemm_ref(A, W, b, BIAS)
        _assert_within(window(Dbuf, Mr), want, err, dtype, ("bias", b is None))
        assert untouched(Dbuf, Mr, torch.full_like(Dbuf, -3.0))

    R0 = _randn((Mr + 3, ldd), 5)
    R = R0.clone()
    G.gemm(A, W, dtype, LS, bias=bias, aux0=gamma, R=window(R, Mr))
    want, err = _gemm_ref(A, W, bias, LS, gamma=gamma, R0=window(R0, Mr))
    _assert_within(window(R, Mr), want, err, torch.float32, "ls_residual")
    assert untouched(R, Mr, R0)

    posbuf = _randn((period, ldd), 6)
    pos = window(posbuf, period)
    rows = Mr + Mr // period
    R0 = torch.full((rows + 3, ldd), 7.0, device=DEV)
    R = R0.clone()
    G.gemm(A, W, dtype, PATCH, bias=bias, aux0=pos, period=period, R=window(R, rows))
    want, err = _gemm_ref(A, W, bias, PATCH, R0=window(R0, rows), pos=pos, period=period)
    _assert_within(window(R, rows), want, err, torch.float32, "patch")
    assert untouched(R, rows, R0)

    # M = 0 (valid pointers; an empty torch view has none): nothing is launched and nothing written
    n0 = L.launch_count()
    D = torch.full((4, N), -3.0, dtype=dtype, device=DEV)
    L.check(L.lib().mdc_gemm(L.ctx(DEV), G.dtype_code(dtype), BIAS, L.ptr(A), A.stride(0), L.ptr(W), W.stride(0), L.ptr(D), D.stride(0),
                             L.ptr(bias), None, 0, 0, N, K, L.stream_ptr()))
    assert L.launch_count() == n0 and torch.equal(D, torch.full_like(D, -3.0))


# ---- strip attention --------------------------------------------------------------------------------------------------------

def _attn_ref(qkv, n_strips, n, H, hd, scale, dim=-1):
    """fp64 softmax(q k^T scale) v (softmax over keys: dim=-1, over queries: dim=-2), the magnitude P @ |V|, and the bound of the
    fp32 arithmetic relative to it: scores carry hd*u*scale*(|q| @ |k|^T) (twice that through exp and the normaliser), the
    P.V sums n*u."""
    q, k, v = [t.reshape(n_strips, n, H, hd).transpose(1, 2).double() for t in qkv.chunk(3, dim=-1)]
    P = torch.softmax(q @ k.transpose(-1, -2) * scale, dim=dim)
    delta = hd * U * scale * (q.abs() @ k.abs().transpose(-1, -2)).amax(dim=(-1, -2), keepdim=True)

    def rows(t):
        return t.transpose(1, 2).reshape(n_strips * n, H * hd)
    mag = P @ v.abs()
    return rows(P @ v), rows(mag), rows((2 * delta + (n + hd) * U) * mag)


def _assert_attn(got, want, mag, err, dtype, what):
    # bf16: the probabilities pass through bf16 on the tensor-core kernels (2^-9 each, 2^-8 with the normaliser) and the output
    # is rounded to bf16
    bound = err + (2.0 ** -8 * mag if dtype == torch.bfloat16 else 0) + OUT_RND[dtype] * want.abs()
    d = (got.double() - want).abs()
    assert (d <= bound).all(), (what, f"max |d| / bound = {(d / bound).max().item():.3g}")


@pytest.mark.parametrize("dtype,n,hd", [(torch.bfloat16, 197, 64), (torch.bfloat16, 300, 64), (torch.bfloat16, 100, 32),
                                        (torch.float32, 197, 64)])
def test_strip_attention_strided_operands_leave_the_rest_untouched(dtype, n, hd):
    """ld_qkv > 3*H*hd, and `out` the view at a 16-byte offset of a wider buffer with rows to spare (tcgen05 kernel at 197 tokens,
    mma.sync at 300, SIMT at head width 32 and in fp32)."""
    n_strips, H, scale = 3, 4, 0.125
    D3 = 3 * H * hd
    qkv = _randn((n_strips * n, D3 + 24), 7).to(dtype)[:, :D3]
    off = 16 // qkv.element_size()
    obuf = torch.full((n_strips * n + 2, H * hd + 16), -5.0, dtype=dtype, device=DEV)
    out = obuf[:n_strips * n, off:off + H * hd]
    G.strip_attention(qkv, n_strips, n, H, hd, scale, out=out)
    want, mag, err = _attn_ref(qkv, n_strips, n, H, hd, scale)
    _assert_attn(out, want, mag, err, dtype, (dtype, n, hd))
    outside = torch.ones_like(obuf, dtype=torch.bool)
    outside[:n_strips * n, off:off + H * hd] = False
    assert torch.equal(obuf[outside], torch.full_like(obuf, -5.0)[outside])


@pytest.mark.parametrize("dtype,n", [(torch.bfloat16, 197), (torch.bfloat16, 256), (torch.bfloat16, 300), (torch.float32, 197)])
def test_strip_attention_softmax_is_sensitive_to_the_scale(dtype, n):
    """One key per query row carries the logit ln(n - 1) and the value 1, every other key logit 0 and value 0: the output is
    p = 1/2 in every channel, and dp/dscale = ln(n - 1) p (1 - p) / scale.  A scale off by 2^-7 moves the output by 1e-2, the
    bound of the arithmetic is 4e-3 in bf16."""
    n_strips, H, hd, scale = 3, 2, 64, 0.125
    qkv = torch.zeros((n_strips, n, 3, H, hd), device=DEV)
    qkv[:, :, 0, :, 0] = 1.0
    top = torch.arange(n_strips) * 37 % n                      # the distinguished key of each strip
    c = torch.log(torch.tensor(n - 1.0)).item() / scale
    qkv[torch.arange(n_strips), top, 1, :, 0] = c
    qkv[torch.arange(n_strips), top, 2] = 1.0
    qkv = qkv.reshape(n_strips * n, 3 * H * hd).to(dtype)
    got = G.strip_attention(qkv, n_strips, n, H, hd, scale)
    want, mag, err = _attn_ref(qkv, n_strips, n, H, hd, scale)
    assert (want - 0.5).abs().max().item() < 0.02
    _assert_attn(got, want, mag, err, dtype, (dtype, n))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n,hd", [(17, 32), (45, 64), (33, 128), (128, 64), (128, 96)])
def test_strip_attention_softmax_over_queries(dtype, n, hd):
    n_strips, H, scale = 2, 3, 0.3
    qkv = _randn((n_strips * n, 3 * H * hd), 8).to(dtype)
    got = G.strip_attention(qkv, n_strips, n, H, hd, scale, soq=1)
    want, mag, err = _attn_ref(qkv, n_strips, n, H, hd, scale, dim=-2)
    _assert_attn(got, want, mag, err, dtype, (dtype, n, hd))


def test_strip_attention_softmax_over_queries_rejects_a_strip_beyond_shared_memory():
    """n = 128 at head width 128 needs (n(n+1) + 3 n hd) * 4 = 262 656 bytes of shared memory, more than a block may have: the
    call is refused with that bound before any CUDA call, and leaves no error behind for the next call."""
    n, H, hd = 128, 2, 128
    qkv = torch.zeros((n, 3 * H * hd), device=DEV)
    with pytest.raises(L.MdcError, match="shared memory"):
        G.strip_attention(qkv, 1, n, H, hd, 0.125, soq=1)
    qkv = _randn((2 * 45, 3 * 4 * 32), 9)
    got = G.strip_attention(qkv, 2, 45, 4, 32, 0.125)
    want, mag, err = _attn_ref(qkv, 2, 45, 4, 32, 0.125)
    _assert_attn(got, want, mag, err, torch.float32, "the call after the rejection")


# ---- LayerNorm --------------------------------------------------------------------------------------------------------------

def _ln_inputs(rows, cols):
    x = _randn((rows, cols), 1) * 3 + 1
    x[1::3] = 1000 + _randn((len(range(1, rows, 3)), cols), 2)      # mean 1000, std 1: a one-pass variance loses it
    w, b = 1 + _randn((cols,), 3, 0.5), _randn((cols,), 4, 0.5)
    want = torch.nn.functional.layer_norm(x.double(), (cols,), w.double(), b.double(), 1e-6)
    return x, w, b, want


def _assert_ln(got, want, dtype, what):
    """Two-pass statistics in fp32: 2e-5 (1 + |want|) on the ordinary rows, 1e-3 on the mean-1000 rows (the fp32 rounding of
    x ~ 1000 is 3e-5, the mean of the row carries ~1e-4); plus the bf16 rounding of the output."""
    tol = torch.full_like(want, 2e-5) * (1 + want.abs())
    tol[1::3] = 1e-3
    if dtype == torch.bfloat16:
        tol = tol + 2.0 ** -8 * want.abs()
    d = (got.double() - want).abs()
    assert (d <= tol).all(), (what, f"max |d| / tol = {(d / tol).max().item():.3g}")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("rows", [1, 2, 777])
@pytest.mark.parametrize("cols", [384, 512, 768, 1024, 256, 260, 2048])
def test_layernorm_paths(cols, rows, dtype):
    """Fast path (row in registers, two rows per warp; 777 rows end in a lone row) at 384 / 512 / 768 / 1024 columns, the
    generic kernel at 256 / 260 / 2048."""
    x, w, b, want = _ln_inputs(rows, cols)
    _assert_ln(G.layernorm(x, w, b, 1e-6, dtype), want, dtype, (cols, rows, dtype))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("cols", [512, 260])
def test_layernorm_into_an_unaligned_strided_output(dtype, cols):
    """ldo % 4 != 0 and `out` one element into its buffer: the generic kernel with scalar stores; neighbours keep their bits."""
    rows = 777
    x, w, b, want = _ln_inputs(rows, cols)
    obuf = torch.full((rows + 1, cols + 6), -9.0, dtype=dtype, device=DEV)
    out = obuf[:rows, 1:1 + cols]
    G.layernorm(x, w, b, 1e-6, dtype, out=out)
    _assert_ln(out, want, dtype, (cols, dtype))
    outside = torch.ones_like(obuf, dtype=torch.bool)
    outside[:rows, 1:1 + cols] = False
    assert torch.equal(obuf[outside], torch.full_like(obuf, -9.0)[outside])


# ---- misaligned operands ----------------------------------------------------------------------------------------------------

def test_misaligned_operands_are_rejected_before_any_launch():
    """Every one of these kernels reads the operand in 8- or 16-byte vectors: a view at a 4- or 8-byte offset is refused by
    the argument checks, and nothing is launched."""
    n0 = L.launch_count()
    buf = torch.zeros(64 * 1024 + 16, device=DEV)
    w, b = torch.ones(512, device=DEV), torch.zeros(512, device=DEV)
    with pytest.raises(L.MdcError):                                   # LayerNorm x at +4 bytes
        G.layernorm(buf[1:1 + 8 * 512].view(8, 512), w, b, 1e-6, torch.float32)
    with pytest.raises(L.MdcError):                                   # fp32 GEMM (FFMA kernel) A at +4 bytes
        G.gemm(buf[1:1 + 64 * 64].view(64, 64), torch.zeros((64, 64), device=DEV), torch.float32, BIAS)
    A16 = torch.zeros((64, 64), dtype=torch.bfloat16, device=DEV)
    R = torch.zeros((66, 64), device=DEV)
    with pytest.raises(L.MdcError):                                   # tensor-core PATCH: positional table at +4 bytes
        G.gemm(A16, A16, torch.bfloat16, PATCH, aux0=buf[1:1 + 32 * 64].view(32, 64), period=32, R=R)
    with pytest.raises(L.MdcError):                                   # SIMT strip attention (fp32, hd 32): qkv at +8 bytes
        G.strip_attention(buf[2:2 + 16 * 96].view(16, 96), 1, 16, 1, 32, 0.125)
    assert L.launch_count() == n0


# ---- the encoder at the bench batch -----------------------------------------------------------------------------------------

def test_encoder_at_the_bench_batch_matches_the_small_batch_path():
    """Config P in bf16 at B = 64 (GEMMs on 256-wide tiles and CTA pairs, PATCH at BN = 256) and, for its first and last images,
    at B = 2 (BN = 64 tiles): both against the fp32 oracle on those two images.  The wide-tile path may not be less accurate."""
    model = cases.build_product_model("P", seed=0, gamma_seed=5)
    sd, cfg = cases.state_dict_of(model), cases.oracle_cfg("P")
    x = cases.images(64, seed=21)
    pick = x[[0, 63]]
    want = O.encoder_forward(sd, pick, cfg)
    model = model.to(DEV).set_precision("bf16")
    e64 = model.encoder(x.to(DEV))[[0, 63]].float().cpu()
    e2 = model.encoder(pick.to(DEV)).float().cpu()
    err64, err2 = (e64 - want).abs().max().item(), (e2 - want).abs().max().item()
    print(f"encoder bf16 vs oracle: B = 64 max|d| = {err64:.3e}, B = 2 max|d| = {err2:.3e}")
    assert err64 <= 1.5 * err2 + 1e-3


# ---- which instantiations ran -----------------------------------------------------------------------------------------------

def _required_gemm_instantiations():
    """gemm_tc_kernel<BN, EPI, EW, F16, CTAS> for every choice gemm_tc_launch can make (EW = 16 only for 256-wide GELU tiles)."""
    ew = lambda bn, e: 16 if (bn == 256 and e == GELU) else 8          # noqa: E731
    req = {(bn, e, ew(bn, e), False, 1) for bn in (64, 128, 256) for e in (BIAS, GELU, RELU, LS, PATCH)}
    req |= {(bn, e, ew(bn, e), False, 2) for bn in (128, 256) for e in (BIAS, GELU, RELU, LS)}
    req |= {(bn, e, 8, True, 1) for bn in (64, 128, 256) for e in (BIAS, RELU)}
    return req


def test_every_required_instantiation_is_reached():
    """Runs the GEMM matrix above plus one call per attention backend and LayerNorm form under torch.profiler and reads the
    kernel names back, so the selection is asserted rather than assumed."""
    if torch.cuda.get_device_properties(DEV).multi_processor_count != 148:
        pytest.skip("the tile selection above is worked out for 148 SMs")
    from torch.profiler import ProfilerActivity, profile
    calls = []
    for case in GEMM_CASES:
        A, W, bias, aux0, R0 = _gemm_operands(case, torch.bfloat16)
        calls.append(lambda c=case, A=A, W=W, bias=bias, aux0=aux0, R0=R0: G.gemm(A, W, torch.bfloat16, c[3], bias=bias, aux0=aux0,
                                                                                period=c[4], R=R0))
    for (Mr, N, K), epi in F16_CASES:
        A, W, bias = _randn((Mr, K), 1, 0.5).half(), _randn((N, K), 2, 0.5).half(), _randn((N,), 3)
        calls.append(lambda A=A, W=W, bias=bias, epi=epi: G.gemm(A, W, torch.float16, epi, bias=bias))
    for dtype, n, hd in ((torch.bfloat16, 197, 64), (torch.bfloat16, 300, 64), (torch.float32, 197, 64), (torch.bfloat16, 100, 32)):
        qkv = _randn((2 * n, 3 * 4 * hd), 7).to(dtype)
        calls.append(lambda qkv=qkv, n=n, hd=hd: G.strip_attention(qkv, 2, n, 4, hd, 0.125))
    for cols in (384, 512, 768, 1024, 260):
        x, w, b, _ = _ln_inputs(64, cols)
        calls.append(lambda x=x, w=w, b=b: G.layernorm(x, w, b, 1e-6, torch.bfloat16))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for call in calls:
            call()
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    gemm = {(int(m[1]), int(m[2]), int(m[3]), m[4] == "true", int(m[5]))
            for s in names for m in [re.search(r"gemm_tc_kernel<(\d+), (\d+), (\d+), (true|false), (\d+)>", s)] if m}
    attn = {m[0] for s in names for m in [re.search(r"attn_umma_kernel|attn_tc_kernel|strip_attn_kernel<\w+, \d+>", s)] if m}
    ln = {m[0] for s in names for m in [re.search(r"layernorm_rows_kernel<[\w:]+, \d+>|layernorm_kernel<[\w:]+>", s)] if m}
    print("\nreached gemm_tc_kernel<BN, EPI, EW, F16, CTAS>:")
    for bn, e, ew, f16, ctas in sorted(gemm):
        print(f"  BN {bn:3d}  {EPI_NAME.get(e, e):12s} EW {ew:2d}  {'fp16' if f16 else 'bf16'}  CTAS {ctas}")
    print("reached attention:", sorted(attn))
    print("reached layernorm:", sorted(ln))
    missing = _required_gemm_instantiations() - gemm
    assert not missing, f"not reached: {sorted(missing)}"
    assert {"attn_umma_kernel", "attn_tc_kernel"} <= attn and any(a.startswith("strip_attn_kernel") for a in attn), attn
    assert {int(re.search(r"(\d+)>$", s)[1]) for s in ln if "rows" in s} == {3, 4, 6, 8} and any("rows" not in s for s in ln), ln
