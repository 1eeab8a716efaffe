"""CPU: the oracle restatement (oracle/mdc_oracle.py) against the golden vectors produced by the
UNMODIFIED reference (oracle/make_golden.py), plus -- when /root/reference is present -- a live
re-check against the reference itself."""
import pytest
import torch

from oracle import cases, mdc_oracle as O, ref_loader

TOL = 2e-5


@pytest.fixture(scope="module")
def case_p():
    pm = cases.build_product_model("P", seed=0, gamma_seed=5)
    return cases.state_dict_of(pm), cases.oracle_cfg("P"), cases.images(2)


def test_encoder_predict_forward_match_reference_golden(case_p, golden):
    sd, cfg, x = case_p
    g = golden("case_P_gamma.pt")
    enc = O.encoder_forward(sd, x, cfg)
    assert (enc - g["enc_out"]).abs().max() < TOL
    assert (O.decoder_predict(sd, enc, g["prefix"], cfg) - g["predict"]).abs().max() < TOL
    assert (O.decoder_forward(sd, enc, g["prefix"][:, 1:], cfg) - g["forward"]).abs().max() < TOL
    # predict's contract: constant BOS row, row L = next-token logits of the prefix (Q5)
    assert torch.all(g["predict"][:, 0] == 300.0)
    assert (O.next_token_logits(sd, enc, g["prefix"], cfg) - g["predict"][:, 4]).abs().max() < TOL


def test_greedy_generate_matches_reference_golden(case_p, golden):
    sd, cfg, x = case_p
    g = golden("case_P_gamma.pt")
    toks, confs, logits = O.generate(sd, x, cfg, max_len=8, return_logits=True)
    assert torch.equal(toks, g["tokens"][:, :9])
    assert (logits - g["logits"][:, :8]).abs().max() < TOL
    assert (torch.stack(confs, 1) - g["confs"][:, :2]).abs().max() < 1e-6


def test_pad_key_bias_is_additive_plus_one(case_p):
    """Q7: a PAD token inside the prefix gets +1.0 on its key, not -inf."""
    sd, cfg, x = case_p
    enc = O.encoder_forward(sd, x[:1], cfg)
    a = O.next_token_logits(sd, enc, torch.tensor([[300, 302, 7]]), cfg)
    cfg2 = cases.oracle_cfg("P"); cfg2.pad_idx = 9999            # no PAD bias at all
    b = O.next_token_logits(sd, enc, torch.tensor([[300, 302, 7]]), cfg2)
    assert (a - b).abs().max() > 1e-3


def test_iou_matches_reference_golden(golden):
    g = golden("case_iou.pt")
    p, q = g["pred"], g["gt"]
    assert torch.equal(O.batch_iou(p, q), g["batch_iou"])
    assert torch.equal(O.batch_max_iou(p, q).flatten(), g["max_iou"])
    assert torch.equal(O.batch_max_iou_torchvision(p, q).flatten(), g["max_iou_tv"])
    assert torch.equal(O.giou_pairwise(p[2], q[2]), g["giou_2"])
    assert torch.equal(O.calculate_iou(p[2], q[2]), g["calc_iou_2"])
    assert torch.isnan(g["calc_iou_zero"]).all() and torch.isnan(O.calculate_iou(p[3], q[4])).all()
    assert abs(O.iou_loss(p[2], q[2]).item() - g["iou_loss_2"].item()) < 1e-6
    assert abs(O.giou_loss_with_scores(p, q)[0].item() - g["giou_loss"].item()) < 1e-6
    # known answers (SURVEY section 4)
    assert abs(g["kat_iou"].item() - 0.14285715) < 1e-7 and abs(g["kat_giou"].item() + 0.07936507) < 1e-7


def test_token_decode_matches_reference_golden(golden):
    """Tokenizer.decode_bboxes / decode restatements against the outputs of the unmodified data_processing.Tokenizer
    (oracle/make_golden.py tokens_case): bit-exact boxes, same labels, same caption ids."""
    g = golden("case_tokens.pt")
    assert torch.equal(O.decode_bboxes(g["tokens"]), g["decode_bboxes"])
    for s, lab, bx, cap in zip(g["tokens"], g["decode_labels"], g["decode_boxes"], g["decode_captions"]):
        olab, obx, ocap = O.decode_sequence(s)
        assert olab == lab and torch.equal(obx, bx)
        assert cap == ("" if ocap is None else [f"w{t}" if 270 <= t < 299 else "<UNK>" for t in ocap])


def test_axial_matches_reference_golden(golden):
    g = golden("case_axial.pt")
    pa = cases.build_product_model("P", seed=2, gamma_seed=7, axial=True)
    sd, cfg = cases.state_dict_of(pa), cases.oracle_cfg("P")
    assert (O.axial_attention(sd, g["xa"], cfg) - g["ax1"]).abs().max() < 1e-6
    assert (O.axial_attention(sd, g["xa"], cfg, axis=-2) - g["ax2"]).abs().max() < 1e-6
    enc = O.encoder_forward(sd, cases.images(2), cfg)
    assert (O.axial_decoder_forward(sd, enc, g["tgt12"], cfg) - g["f12"]).abs().max() < TOL


def test_top_k_top_p_restatement_against_transformers_warpers():
    """Q2: the removed helper is restated; cross-check with the warpers that still exist."""
    tr = pytest.importorskip("transformers.generation.logits_process")
    torch.manual_seed(3)
    logits = torch.randn(5, 305)
    ids = torch.zeros(5, 1, dtype=torch.long)
    for k, p in [(5, 1.0), (0, 0.9), (7, 0.8), (1, 1.0)]:
        want = logits.clone()
        if k > 0:
            want = tr.TopKLogitsWarper(top_k=k)(ids, want)
        if p < 1.0:
            want = tr.TopPLogitsWarper(top_p=p)(ids, want)
        got = O.top_k_top_p_filtering(logits, top_k=k, top_p=p)
        assert torch.equal(torch.isinf(got), torch.isinf(want)), (k, p)


def test_adaptive_pool_and_interp_restatements():
    x = torch.randn(2, 5, 512)
    for out in (256, 1024, 64, 300):
        assert torch.allclose(O.adaptive_avg_pool_channels(x, out), torch.nn.functional.adaptive_avg_pool1d(x, out), atol=1e-6)
    pos = torch.randn(1, 99, 16)
    for n in (5, 13, 99, 150):
        want = torch.nn.functional.interpolate(pos.permute(0, 2, 1), size=n, mode="linear", align_corners=False).permute(0, 2, 1)
        assert torch.allclose(O.interp_pos_embed(pos, n), want, atol=1e-6)


def test_live_reference_agrees_with_oracle(case_p, golden):
    """EncoderDecoder.predict of the unmodified reference on one image against the oracle: always against the reference's
    committed output for that image (case_P_gamma.pt, image 0 of the same prefix batch), and against a live run of the
    reference too where its source tree is present (oracle/ref_loader.py).  The stored half checks the same composition
    (encoder, then decoder predict) as test_encoder_predict_forward_match_reference_golden, here at batch size one."""
    sd, cfg, x = case_p
    got = O.model_predict(sd, x[:1], cases.PREFIX[:1], cfg)
    assert (got - golden("case_P_gamma.pt")["predict"][:1]).abs().max() < TOL
    if not ref_loader.available():
        return
    R = ref_loader.load()
    with cases.quiet():
        enc = R["model"].Encoder(model_name=cases.VIT, pretrained=False, out_dim=256)
        dec = R["model"].Decoder(305, 196, 256, 8, 6)
        rm = R["model"].EncoderDecoder(enc, dec).eval()
    rm.load_state_dict(sd)
    with torch.no_grad(), cases.quiet():
        want = rm.predict(x[:1], cases.PREFIX[:1])
    assert (got - want).abs().max() < TOL


def test_preprocess_restatement_against_cv2_goldens(golden):
    """oracle.cv2_resize_linear_u8 (integer restatement of cv2.resize INTER_LINEAR on uint8, the A.Resize step of
    inference_p.py:148-158) against the committed outputs of the real cv2 -- and against the live cv2 where it is installed."""
    import numpy as np
    g = golden("case_preprocess.pt")
    for name, src, size in (("gray", g["gray"], 224), ("bgr", g["bgr"], 224), ("small", g["small"], 224), ("big", g["big"], 224),
                            ("gray320", g["gray"][:1], 320)):
        for im, want in zip(src.numpy(), g["resized_" + name].numpy()):
            rgb = im if im.ndim == 2 else np.ascontiguousarray(im[..., ::-1])
            assert np.array_equal(O.cv2_resize_linear_u8(rgb, size, size), want), name
    try:
        import cv2
    except ImportError:
        return
    rng = np.random.default_rng(3)
    for h, w, size, c in ((200, 200, 224, 1), (199, 201, 224, 3), (448, 448, 224, 3), (37, 53, 512, 1)):
        im = rng.integers(0, 256, (h, w) if c == 1 else (h, w, c), dtype=np.uint8)
        assert np.array_equal(O.cv2_resize_linear_u8(im, size, size), cv2.resize(im, (size, size), interpolation=cv2.INTER_LINEAR))


def test_metric_restatements_known_answers():
    """mAP / BLEU restatements (third-party arithmetic absent: parity unpinned) on answers known in closed form."""
    import mdcnet_b200 as M
    gb = torch.tensor([[0., 0, 10, 10], [20, 20, 40, 40]]); gl = torch.tensor([1, 2])
    perfect = [{"boxes": gb.clone(), "scores": torch.tensor([0.9, 0.8]), "labels": gl.clone()}]
    assert abs(O.mean_average_precision(perfect, [{"boxes": gb, "labels": gl}]) - 1.0) < 1e-12
    # one true positive ranked below one false positive of the same class: precision 1/2 at every recall level
    p = [{"boxes": torch.tensor([[100., 100, 110, 110], [0, 0, 10, 10]]), "scores": torch.tensor([0.9, 0.5]), "labels": torch.tensor([1, 1])}]
    assert abs(O.mean_average_precision(p, [{"boxes": gb[:1], "labels": gl[:1]}]) - 0.5) < 1e-9
    ref = "the surface shows a long scratch".split()
    assert M.calculate_bleu_scores([ref], [ref]) == [1.0]
    assert M.calculate_bleu_scores([ref], [["unrelated"]]) == [0.0]
    got = M.calculate_bleu_scores([list("abcde")], [list("abxde")])[0]
    assert abs(got - (0.8 * 0.5 * (0.1 / 3) * (0.1 / 2)) ** 0.25) < 1e-12           # method1: zero counts -> epsilon 0.1
