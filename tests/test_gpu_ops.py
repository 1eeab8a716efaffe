"""GPU: every kernel behind the C ABI against a plain fp32/fp64 torch statement of the same op (and
the reference-derived golden vectors for IoU).  Tolerances are stated per test."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

import mdcnet_b200 as M  # noqa: E402
from oracle import cases, mdc_oracle as O  # noqa: E402
from tests import gpu_util as G  # noqa: E402

L = M._lib
DEV = "cuda"

# (M, N, K): the encoder/decoder GEMM shapes of SURVEY 2.1 at small batch, ragged tails, and skinny cases
GEMM_SHAPES = [(392, 512, 768), (394, 1536, 512), (394, 512, 512), (394, 2048, 512), (394, 512, 2048), (392, 512, 256),
               (1, 512, 512), (127, 64, 64), (129, 72, 128), (300, 136, 192), (2000, 1536, 512)]


def _mk(shape, dtype, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(shape, generator=g) * 0.5).to(DEV, dtype)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", GEMM_SHAPES)
def test_gemm_bias_epilogues(dtype, shape):
    Mr, N, K = shape
    A, W = _mk((Mr, K), dtype, 1), _mk((N, K), dtype, 2)
    bias = _mk((N,), torch.float32, 3)
    ref = A.double() @ W.double().T + bias.double()
    # fp32: FFMA, K-ordered accumulation -> 1e-4 abs at |ref| ~ sqrt(K)/4; bf16: inputs exact in bf16, fp32 accumulate,
    # output rounded to bf16 (rel 2^-8)
    for epi, fn in [(L.EPI_BIAS, lambda r: r), (L.EPI_BIAS_RELU, torch.relu),
                    (L.EPI_BIAS_GELU, lambda r: torch.nn.functional.gelu(r))]:
        D = G.gemm(A, W, dtype, epi, bias=bias)
        want = fn(ref)
        err = (D.double() - want).abs().max().item()
        tol = 2e-4 if dtype == torch.float32 else 2e-2 + want.abs().max().item() * 2 ** -8
        assert err <= tol, (shape, dtype, epi, err, tol)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_gemm_layerscale_residual_and_patch_epilogues(dtype):
    Mr, N, K = 394, 512, 2048
    A, W = _mk((Mr, K), dtype, 1), _mk((N, K), dtype, 2)
    bias, gamma = _mk((N,), torch.float32, 3), _mk((N,), torch.float32, 4)
    R0 = _mk((Mr, N), torch.float32, 5)
    R = R0.clone()
    G.gemm(A, W, dtype, L.EPI_LS_RESIDUAL, bias=bias, aux0=gamma, R=R)
    want = R0.double() + gamma.double() * (A.double() @ W.double().T + bias.double())
    assert (R.double() - want).abs().max().item() < (5e-4 if dtype == torch.float32 else 5e-3)
    # patch epilogue: 2 images x 196 patches -> rows shifted past each image's cls slot, + pos
    Mr, K = 392, 768
    A, W = _mk((Mr, K), dtype, 6), _mk((N, K), dtype, 7)
    pos = _mk((196, N), torch.float32, 8)
    R = torch.full((2 * 197, N), 7.0, dtype=torch.float32, device=DEV)
    G.gemm(A, W, dtype, L.EPI_PATCH, bias=bias, aux0=pos, period=196, R=R)
    want = (A.double() @ W.double().T + bias.double()).reshape(2, 196, N) + pos.double()
    got = R.reshape(2, 197, N)
    assert torch.all(got[:, 0] == 7.0)                      # cls rows untouched
    assert (got[:, 1:].double() - want).abs().max().item() < (5e-4 if dtype == torch.float32 else 5e-3)


@pytest.mark.parametrize("shape,epi", [((12608, 1536, 512), "bias"), ((12608, 2048, 512), "gelu"), ((12608, 512, 2048), "residual"),
                                       ((12608, 512, 512), "residual"), ((9999, 2048, 512), "gelu")])
def test_gemm_encoder_shapes_at_the_bench_batch(shape, epi):
    """The encoder GEMMs at B = 64 -- the shapes that run as CTA pairs (tcgen05.mma.cta_group::2, 256 x 256 tiles, several tile waves per
    CTA, a ragged last row pair) -- against fp64 on the same bf16 operands."""
    Mr, N, K = shape
    A, W = _mk((Mr, K), torch.bfloat16, 11), _mk((N, K), torch.bfloat16, 12) * 0.2
    bias = _mk((N,), torch.float32, 13)
    ref = A.double() @ W.double().T + bias.double()
    if epi == "residual":
        gamma, R0 = _mk((N,), torch.float32, 14), _mk((Mr, N), torch.float32, 15)
        R = R0.clone()
        G.gemm(A, W, torch.bfloat16, L.EPI_LS_RESIDUAL, bias=bias, aux0=gamma, R=R)
        want = R0.double() + gamma.double() * ref
        assert (R.double() - want).abs().max().item() < 5e-3
    else:
        D = G.gemm(A, W, torch.bfloat16, L.EPI_BIAS_GELU if epi == "gelu" else L.EPI_BIAS, bias=bias)
        want = torch.nn.functional.gelu(ref) if epi == "gelu" else ref
        err = (D.double() - want).abs()
        assert (err <= 1e-3 + want.abs() * 2 ** -8).all(), err.max().item()


def test_gemm_gelu_epilogue_is_the_exact_erf_form_to_output_rounding():
    """GELU in the epilogue is max(x,0) - a 2^q(a) with a fitted polynomial q (|error| <= 3e-7, tools/gelu_fit.py): on a dense sweep of
    x in [-9, 9] the bf16 result must be the correctly rounded exact-erf GELU up to one unit in the last place of bf16."""
    Mr, N, K = 8192, 64, 64
    x = torch.linspace(-9, 9, Mr, device=DEV).to(torch.bfloat16)
    A = torch.zeros((Mr, K), dtype=torch.bfloat16, device=DEV); A[:, 0] = x
    W = torch.zeros((N, K), dtype=torch.bfloat16, device=DEV); W[:, 0] = 1
    D = G.gemm(A, W, torch.bfloat16, L.EPI_BIAS_GELU, bias=torch.zeros(N, device=DEV))
    want = torch.nn.functional.gelu(x.double())
    got = D[:, 0].double()
    assert torch.equal(D[:, 0], D[:, N - 1])
    assert ((got - want).abs() <= want.abs() * 2 ** -8 + 1e-6).all(), (got - want).abs().max().item()
    # and against the correctly rounded value: equal almost everywhere (ties of the rounding can differ by one ulp)
    # (where |GELU| > 1e-5, i.e. x > -4.4: below that the value is the difference of float32 roundings and, for x < -6, the clamp a <= 6)
    exact_bf16 = want.to(torch.bfloat16)
    sel = want.abs() > 1e-5
    assert (D[:, 0][sel] == exact_bf16[sel]).float().mean().item() > 0.995


def test_gemm_tcgen05_matches_ffma_on_same_bf16_inputs():
    """The tensor-core kernel and the FFMA kernel see identical bf16 operands; only the summation order differs."""
    A, W = _mk((1000, 512), torch.bfloat16, 1), _mk((1536, 512), torch.bfloat16, 2)
    ref = (A.float() @ W.float().T)
    D = G.gemm(A, W, torch.bfloat16, L.EPI_BIAS)
    assert (D.float() - ref).abs().max().item() <= ref.abs().max().item() * 2 ** -7


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_layernorm(dtype):
    x = _mk((777, 512), torch.float32, 1) * 3 + 1
    w, b = _mk((512,), torch.float32, 2), _mk((512,), torch.float32, 3)
    got = G.layernorm(x, w, b, 1e-6, dtype)
    want = torch.nn.functional.layer_norm(x.double(), (512,), w.double(), b.double(), 1e-6)
    assert (got.double() - want).abs().max().item() < (2e-5 if dtype == torch.float32 else 3e-2)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("cfg", [(3, 197, 8, 64, 0.125), (2, 99, 8, 32, 0.125), (28, 14, 8, 64, 0.125), (2, 17, 2, 128, 0.3),
                                 (1, 1025, 8, 64, 0.125), (2, 300, 8, 64, 0.125), (2, 208, 8, 64, 0.125), (2, 209, 8, 64, 0.125), (5, 1, 8, 32, 0.125),
                                 # bf16 head width 64: the mma.sync kernel below 16 and above 256 tokens, the tcgen05 kernel at its bounds
                                 (3, 1, 4, 64, 0.125), (3, 7, 4, 64, 0.125), (3, 15, 4, 64, 0.125), (3, 16, 4, 64, 0.125),
                                 (2, 255, 4, 64, 0.125), (2, 256, 4, 64, 0.125), (2, 257, 4, 64, 0.125),
                                 # many waves: the bench's 64 strips and config 5's 256 strips of 197 tokens
                                 (64, 197, 8, 64, 0.125), (256, 197, 8, 64, 0.125),
                                 # head widths 32 and 128 with keys over several 64-key tiles
                                 (2, 300, 4, 32, 0.125), (2, 300, 2, 128, 0.125)])
def test_strip_attention(dtype, cfg):
    n_strips, n, H, hd, scale = cfg
    qkv = _mk((n_strips * n, 3 * H * hd), dtype, 4)
    got = G.strip_attention(qkv, n_strips, n, H, hd, scale)
    q, k, v = [t.reshape(n_strips, n, H, hd).transpose(1, 2).double() for t in qkv.chunk(3, dim=-1)]
    want = (torch.softmax(q @ k.transpose(-1, -2) * scale, dim=-1) @ v).transpose(1, 2).reshape(n_strips * n, H * hd)
    assert (got.double() - want).abs().max().item() < (2e-5 if dtype == torch.float32 else 1.5e-2)


def test_strip_attention_softmax_over_queries():
    n_strips, n, H, hd = 2, 17, 8, 32
    qkv = _mk((n_strips * n, 3 * H * hd), torch.float32, 5)
    got = G.strip_attention(qkv, n_strips, n, H, hd, 0.125, soq=1)
    q, k, v = [t.reshape(n_strips, n, H, hd).transpose(1, 2).double() for t in qkv.chunk(3, dim=-1)]
    want = (torch.softmax(q @ k.transpose(-1, -2) * 0.125, dim=-2) @ v).transpose(1, 2).reshape(n_strips * n, H * hd)
    assert (got.double() - want).abs().max().item() < 2e-5


def test_iou_kernels_bit_exact_against_reference_golden(golden):
    g = golden("case_iou.pt")
    p, q = g["pred"].to(DEV), g["gt"].to(DEV)
    got = torch.stack(M.calculate_batch_iou(p, q)).cpu()
    assert torch.equal(got, g["batch_iou"])                                  # bit-exact (contract: 1e-6)
    assert torch.equal(torch.tensor(M.calculate_batch_max_iou(p, q)), g["max_iou"])
    assert torch.equal(torch.tensor(M.calculate_batch_max_iou_torchvision(p, q)), g["max_iou_tv"])
    assert torch.equal(M.giou_pairwise(p[2], q[2]).cpu(), g["giou_2"])
    assert torch.equal(M.calculate_iou(p[2], q[2]).cpu(), g["calc_iou_2"])
    assert torch.isnan(M.calculate_iou(p[3], q[4])).all()
    assert abs(M.iou_loss(p[2], q[2]).item() - g["iou_loss_2"].item()) < 1e-6
    loss, scores = M.giou_loss_with_scores(p, q)
    assert abs(loss.item() - g["giou_loss"].item()) < 1e-6
    assert len(scores) == len(g["giou_scores"])
    for a, b in zip(scores, g["giou_scores"]):
        assert a.shape == b.shape and (a.numel() == 0 or (a.cpu() - b).abs().max() < 1e-6)
    assert abs(M.bbox_iou(torch.tensor([[0., 0, 10, 10]], device=DEV), torch.tensor([[5., 5, 15, 15]], device=DEV)).item() - 0.14285715) < 1e-7


def test_iou_full_size_properties():
    """BASELINE config 5 size (B=256, N<=19, M=5) and beyond: symmetry, self-IoU, range, oracle agreement."""
    B, N, Mg = 4096, 19, 5
    g = torch.Generator().manual_seed(3)
    p = torch.rand(B, N, 4, generator=g) * 160; p[..., 2:] = p[..., :2] + 8 + torch.rand(B, N, 2, generator=g) * 56
    q = torch.rand(B, Mg, 4, generator=g) * 160; q[..., 2:] = q[..., :2] + 8 + torch.rand(B, Mg, 2, generator=g) * 56
    p[::7, 10:] = 0; q[::5, 3:] = 0
    got = torch.stack(M.calculate_batch_iou(p.to(DEV), q.to(DEV))).cpu()
    assert torch.equal(got, O.batch_iou(p, q))
    rev = torch.stack(M.calculate_batch_iou(q.to(DEV), p.to(DEV))).cpu()
    assert torch.equal(rev, got.transpose(1, 2))
    assert got.min() >= 0 and got.max() <= 1
    self_iou = torch.stack(M.calculate_batch_iou(q.to(DEV), q.to(DEV))).cpu()
    d = torch.diagonal(self_iou, dim1=1, dim2=2)
    assert torch.all((d > 0.999999) | (q.abs().sum(-1) == 0))
    # empty batch edge cases
    assert M.calculate_batch_max_iou(torch.zeros(2, 0, 4, device=DEV), torch.zeros(2, 3, 4, device=DEV)) == []


def test_iou_shapes_beyond_the_shared_memory_staging():
    """Shapes the reference accepts whose GT / output staging does not fit shared memory take the kernel's direct form:
    bbox_iou((300,4),(300,4)); calculate_batch_max_iou_torchvision with pred (B,1,4) and 64 GT boxes per image (N = 1)."""
    g = torch.Generator().manual_seed(8)
    def boxes(*shape):
        b = torch.rand(*shape, 4, generator=g) * 160; b[..., 2:] = b[..., :2] + 8 + torch.rand(*shape, 2, generator=g) * 56
        return b
    a, b = boxes(300), boxes(300)
    assert torch.equal(M.bbox_iou(a.to(DEV), b.to(DEV)).cpu(), O.bbox_iou(a, b))
    p, q = boxes(37, 1), boxes(37, 64)
    q[::4, 50:] = 0
    assert torch.equal(torch.tensor(M.calculate_batch_max_iou_torchvision(p.to(DEV), q.to(DEV))), O.batch_max_iou_torchvision(p, q).flatten())
    assert torch.equal(torch.stack(M.calculate_batch_iou(p.to(DEV), q.to(DEV))).cpu(), O.batch_iou(p, q))
    p2, q2 = boxes(2, 3), boxes(2, 700)                    # B = 2: the staging is sized for the images a block touches, not 258
    assert torch.equal(torch.stack(M.calculate_batch_iou(p2.to(DEV), q2.to(DEV))).cpu(), O.batch_iou(p2, q2))


def test_select_greedy_topk_topp_against_oracle():
    torch.manual_seed(0)
    logits = torch.randn(64, 305) * 3
    logits[5, 17] = logits[5, 200] = logits[5].max() + 1          # tie -> first index
    tok, conf = G.select(logits.to(DEV))
    assert torch.equal(tok.cpu().long(), logits.argmax(-1))
    assert tok[5].item() == 17
    assert (conf.cpu() - torch.softmax(logits, -1).max(-1)[0]).abs().max() < 1e-6
    u = torch.rand(64)
    for k, p in [(5, 1.0), (0, 0.9), (7, 0.8), (1, 1.0), (305, 1.0)]:
        filt = O.top_k_top_p_filtering(logits, top_k=k, top_p=p)
        want = O.sample_from_uniform(filt, u)
        tok, conf = G.select(logits.to(DEV), top_k=k, top_p=p, uniforms=u.to(DEV))
        assert torch.equal(tok.cpu().long(), want), (k, p)
        assert (conf.cpu() - torch.softmax(filt, -1).max(-1)[0]).abs().max() < 1e-6


def test_preprocess_is_bit_exact_against_cv2_goldens(golden):
    """SURVEY 8f row 2: the fused transform kernel against tests/golden/case_preprocess.pt -- uint8 outputs of the REAL
    cv2.resize(INTER_LINEAR) (what A.Resize runs on the reference's uint8 images, inference_p.py:148-158) for gray, BGR colour,
    strong upscaling, downscaling and a second model size.  Integer work: the kernel's float32 output must be EXACTLY A.Normalize
    of cv2's uint8 pixels (torch.equal), i.e. the uint8 rounding is reproduced bit for bit."""
    g = golden("case_preprocess.pt")
    import numpy as np
    for name, src, size in (("gray", g["gray"], 224), ("bgr", g["bgr"], 224), ("small", g["small"], 224), ("big", g["big"], 224),
                            ("gray320", g["gray"][:1], 320)):
        r = g["resized_" + name].numpy()
        want = torch.stack([torch.from_numpy(O.albu_normalize(np.repeat(im[:, :, None], 3, axis=2) if im.ndim == 2 else im)).permute(2, 0, 1)
                            for im in r])
        got = (M.preprocess_gray if src.dim() == 3 else M.preprocess_bgr)(src.to(DEV), size=size).cpu()
        assert got.shape == want.shape and torch.equal(got, want), name
        # and the uint8 pixel recovered from the kernel's output is cv2's
        mean = torch.tensor(O.IMAGENET_MEAN).view(1, 3, 1, 1) * 255.0; std = torch.tensor(O.IMAGENET_STD).view(1, 3, 1, 1) * 255.0
        px = torch.round(got * std + mean).to(torch.uint8).permute(0, 2, 3, 1)
        assert torch.equal(px[..., 0] if src.dim() == 3 else px, g["resized_" + name]), name
    out = torch.empty((3, 3, 224, 224), dtype=torch.float32, device=DEV)
    u8 = O.synth_gray_u8(3, hw=200, seed=9).to(DEV)
    L.check(L.lib().mdc_preprocess_gray(L.ctx(DEV), L.ptr(u8), 3, 200, 200, L.ptr(out), 224, L.stream_ptr()))      # through the C ABI
    assert torch.equal(out.cpu(), O.preprocess_u8(u8.cpu()))


def test_interp_rows():
    pos = torch.randn(1, 99, 256)
    for n in (5, 13, 150, 257):
        got = torch.empty((n, 256), dtype=torch.float32, device=DEV)
        src = pos[0].to(DEV).contiguous()
        L.check(L.lib().mdc_interp_rows(L.ctx(DEV), L.ptr(src), 99, L.ptr(got), n, 256, L.stream_ptr()))
        assert (got.cpu() - O.interp_pos_embed(pos, n)[0]).abs().max().item() < 1e-6


def test_bad_arguments_fail_loudly():
    A = torch.zeros((4, 6), device=DEV)
    with pytest.raises(L.MdcError):
        G.gemm(A, A, torch.float32, L.EPI_BIAS)          # K % 4 != 0
    with pytest.raises(L.MdcError):
        G.strip_attention(torch.zeros((4, 3 * 8 * 24), device=DEV), 1, 4, 8, 24, 1.0)   # head_dim unsupported


def test_token_decode_kernel_bit_exact_against_reference_golden(golden):
    """csrc/tokens.cu through the host mirror against the unmodified reference Tokenizer's outputs (tests/golden/case_tokens.pt)."""
    g = golden("case_tokens.pt")
    tk = M.Tokenizer(num_bins=224, width=224, height=224, vocab={i: f"w{i}" for i in range(270, 299)})
    toks = g["tokens"].to(DEV)
    bb = tk.decode_bboxes(toks)
    assert bb.is_cuda and bb.shape == g["decode_bboxes"].shape and torch.equal(bb.cpu(), g["decode_bboxes"])
    labels, boxes, counts, cap, cap_len = tk.decode_batch(toks)
    for i in range(toks.shape[0]):
        n = int(counts[i])
        assert labels[i, :n].tolist() == g["decode_labels"][i]
        assert torch.equal(boxes[i, :n].cpu(), g["decode_boxes"][i])
        assert boxes[i, n:].abs().sum() == 0
        lab1, bx1, cap1 = tk.decode(toks[i])                     # the single-sequence entry point of the reference
        assert lab1 == g["decode_labels"][i] and cap1 == g["decode_captions"][i]
        assert torch.equal(torch.tensor(bx1).reshape(-1, 4).float(), g["decode_boxes"][i])


def test_token_decode_kernel_full_size_against_oracle():
    """Config 5 shape: B=256 sequences of 257 tokens (random grammar soup), both modes, bit-exact against the CPU oracle."""
    gen = torch.Generator().manual_seed(5)
    B, Ln = 256, 257
    toks = torch.randint(0, 305, (B, Ln), generator=gen)
    # make labels / markers frequent enough that boxes actually appear
    pick = torch.rand((B, Ln), generator=gen)
    toks = torch.where(pick < 0.15, torch.randint(258, 268, (B, Ln), generator=gen), toks)
    toks = torch.where((pick >= 0.15) & (pick < 0.6), torch.randint(0, 226, (B, Ln), generator=gen), toks)
    toks[:, 0] = 300; toks[::2, 5] = 303; toks[::2, 9] = 304; toks[::5, 200] = 301
    tk = M.Tokenizer(num_bins=224, width=224, height=224)
    bb = tk.decode_bboxes(toks.to(DEV)).cpu()
    want = O.decode_bboxes(toks)
    assert bb.shape == want.shape and torch.equal(bb, want)
    labels, boxes, counts, cap, cap_len = tk.decode_batch(toks.to(DEV))
    for i in range(0, B, 7):
        olab, obx, ocap = O.decode_sequence(toks[i])
        n = int(counts[i])
        assert labels[i, :n].tolist() == olab and torch.equal(boxes[i, :n].cpu(), obx)
        assert (int(cap_len[i]) == -1) if ocap is None else (cap[i, :int(cap_len[i])].tolist() == ocap)


def test_postprocess_batched_equals_per_sample_decode(golden):
    g = golden("case_tokens.pt")
    tk = M.Tokenizer(num_bins=224, width=224, height=224, vocab={i: f"w{i}" for i in range(270, 299)})
    toks = g["tokens"]
    confs = [torch.full((toks.shape[0],), 0.5 + 0.01 * j) for j in range(25)]
    bboxes, labels, caps, cf = M.postprocess_with_captions(toks, confs, tk)
    b3, l3, c3 = M.postprocess(toks, confs, tk)            # the call site of inference_p.py:225 unpacks three lists
    assert b3 == bboxes and l3 == labels and c3 == cf
    eos = (toks == 301).float().argmax(-1)
    for i in range(toks.shape[0]):
        e = int(eos[i])
        if e == 0 or (e - 1) % 5 != 0:
            assert bboxes[i] is None and labels[i] is None
            continue
        assert labels[i] == g["decode_labels"][i] and caps[i] == g["decode_captions"][i]
        assert torch.equal(torch.tensor(bboxes[i]).reshape(-1, 4).float(), g["decode_boxes"][i])
        assert len(cf[i]) == len(bboxes[i])


def test_top_k_sampling_helpers_against_oracle():
    """data_processing.py:786-835 top_k_sampling / top_k_sampling_with_scores_2d with shared uniforms: same indices as the oracle's
    inverse-CDF draw over the top-k-filtered softmax, same probabilities to 1e-6."""
    gen = torch.Generator().manual_seed(12)
    logits = torch.randn(64, 305, generator=gen) * 2.0
    logits[3, 10] = logits[3, 20] = logits[3].max() + 1.0           # a tie inside the top-k
    u = torch.rand(64, generator=gen)
    idx, score = M.top_k_sampling_with_scores_2d(logits.to(DEV), 5, uniforms=u.to(DEV))
    idx1 = M.top_k_sampling(logits.to(DEV), 5, uniforms=u.to(DEV))
    filt = O.top_k_top_p_filtering(logits.clone(), top_k=5, top_p=1.0)
    want = O.sample_from_uniform(filt, u)
    probs = torch.softmax(filt, dim=-1)
    assert idx.shape == (64, 1) and idx.dtype == torch.int64 and torch.equal(idx.cpu().view(-1), want.view(-1)) and torch.equal(idx, idx1)
    assert (score.cpu().view(-1) - probs.gather(1, want.view(-1, 1)).view(-1)).abs().max().item() < 1e-6


def _det_case(seed, B=40, classes=6):
    g = torch.Generator().manual_seed(seed)
    preds, targets = [], []
    for i in range(B):
        m = int(torch.randint(0, 6, (1,), generator=g))
        gb = torch.rand(m, 4, generator=g) * 160; gb[:, 2:] = gb[:, :2] + 8 + torch.rand(m, 2, generator=g) * 56
        gl = torch.randint(0, classes, (m,), generator=g)
        n = int(torch.randint(0, 12, (1,), generator=g))
        pb = torch.rand(n, 4, generator=g) * 160; pb[:, 2:] = pb[:, :2] + 8 + torch.rand(n, 2, generator=g) * 56
        pl = torch.randint(0, classes, (n,), generator=g)
        k = min(n, m)
        if k:                                       # some predictions are jittered copies of ground-truth boxes (true positives)
            pb[:k] = gb[:k] + torch.randn(k, 4, generator=g) * 6; pl[:k] = gl[:k]
        ps = torch.rand(n, generator=g)
        if n > 3:
            ps[1] = ps[3]                           # a score tie: the stable order decides
        preds.append({"boxes": pb, "scores": ps, "labels": pl}); targets.append({"boxes": gb, "labels": gl})
    return preds, targets


def test_map_matching_kernel_and_accumulation_against_the_restated_coco_evaluation():
    """SURVEY 8f row 4: MeanAveragePrecision (train_val_epoch.py:205-231, iou_thresholds = [0.3]) -- batched matching kernel +
    host accumulation against the oracle's plain-Python restatement of COCOeval (parity unpinned: torchmetrics is absent)."""
    for seed in (1, 2, 3):
        preds, targets = _det_case(seed)
        m = M.MeanAveragePrecision(box_format="xyxy", iou_thresholds=[0.3], class_metrics=True).to(DEV)
        for p, t in zip(preds, targets):
            if p["scores"].nelement() == 0:        # the reference's empty-prediction form (train_val_epoch.py:219-225)
                p = {"boxes": torch.empty((0, 4)), "scores": torch.empty((0,)), "labels": torch.empty((0,), dtype=torch.int64)}
            m.update([p], [t])
        got = m.compute()
        want = O.mean_average_precision(preds, targets, iou_thresholds=(0.3,))
        assert abs(got["map"].item() - want) < 1e-6, (seed, got["map"].item(), want)      # the result tensor is float32, like torchmetrics'
        assert got["map_per_class"].numel() == got["classes"].numel()
    # known answers: perfect predictions -> 1, disjoint predictions -> 0, several thresholds -> their mean
    gb = torch.tensor([[0., 0, 10, 10], [20, 20, 40, 40]]); gl = torch.tensor([1, 2])
    m = M.MeanAveragePrecision(iou_thresholds=[0.3]).to(DEV)
    m.update([{"boxes": gb.clone(), "scores": torch.tensor([0.9, 0.8]), "labels": gl.clone()}], [{"boxes": gb, "labels": gl}])
    assert abs(m.compute()["map"].item() - 1.0) < 1e-6
    m = M.MeanAveragePrecision(iou_thresholds=[0.3]).to(DEV)
    m.update([{"boxes": gb + 100, "scores": torch.tensor([0.9, 0.8]), "labels": gl.clone()}], [{"boxes": gb, "labels": gl}])
    assert m.compute()["map"].item() == 0.0
    preds, targets = _det_case(9)
    m = M.MeanAveragePrecision(iou_thresholds=[0.3, 0.5, 0.75]).to(DEV)
    m.update(preds, targets)
    assert abs(m.compute()["map"].item() - O.mean_average_precision(preds, targets, iou_thresholds=(0.3, 0.5, 0.75))) < 1e-6
