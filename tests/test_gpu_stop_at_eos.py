"""GPU: stop at EOS (generate(..., stop_at_eos=True), generate_tokens(..., eos_token=...), mdc_decode_state.stop_at_eos).

The models make EOS arrive at varied, predictable steps without any test hook: the no-stop run of the unmodified model gives, per
image and step, the margin max_{v != eos} logit_v - logit_eos; adding a constant delta to the EOS bias makes an image emit EOS at the
first step whose margin is below delta (the trajectory before that step is unchanged).  delta is chosen so that some images finish
at spread-out steps and some never do, and so that no margin lies within 1e-3 of it (no near-ties).  The contract is then checked
between the stop and the no-stop runs of the modified model."""

import pytest
import torch

pytestmark = pytest.mark.gpu

import mdcnet_b200 as M  # noqa: E402
from oracle import cases  # noqa: E402
from tests.eos_helpers import EOS, choose_delta, eos_bias  # noqa: E402

DEV = "cuda"
PAD, BOS = 302, 300


@pytest.fixture(scope="module")
def model_p():
    return cases.build_product_model("P", seed=0, gamma_seed=5).to(DEV)


def _model_t():
    cases.product_cfg(100)
    torch.manual_seed(4)
    enc = M.Encoder(model_name=cases.VIT, pretrained=False, out_dim=1024)
    dec = M.Decoder(332, 196, 1024, 8, 8)
    model = M.EncoderDecoder(enc, dec).eval()
    g = torch.Generator().manual_seed(9)
    with torch.no_grad():
        for k, p in model.named_parameters():
            if k.endswith("gamma"):
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)
    return model.to(DEV)


def check_contract(tok_ns, conf_ns, tok_s, conf_s, T):
    """Every bullet of the stop-at-EOS contract, stop run (tok_s, conf_s) against no-stop run (tok_ns, conf_ns).  Returns the e_b."""
    tok_ns, conf_ns, tok_s, conf_s = tok_ns.cpu(), conf_ns.cpu(), tok_s.cpu(), conf_s.cpu()
    assert tok_s.shape == tok_ns.shape == (tok_ns.shape[0], T + 1) and conf_s.shape == conf_ns.shape == (tok_ns.shape[0], (T + 3) // 4)
    firsts = []
    for b in range(tok_ns.shape[0]):
        hits = (tok_ns[b, 1:] == EOS).nonzero()
        if len(hits) == 0:
            assert torch.equal(tok_s[b], tok_ns[b]) and torch.equal(conf_s[b], conf_ns[b]), b
            firsts.append(None)
            continue
        e = int(hits[0])
        assert torch.equal(tok_s[b, :e + 2], tok_ns[b, :e + 2]), (b, e)
        assert (tok_s[b, e + 2:] == PAD).all(), (b, e, tok_s[b])
        assert torch.equal(conf_s[b, :e // 4 + 1], conf_ns[b, :e // 4 + 1]), (b, e)
        assert (conf_s[b, e // 4 + 1:] == 0).all(), (b, e)
        firsts.append(e)
    # postprocess cuts at the first EOS already: the same boxes, labels, captions and confidences
    tok = M.Tokenizer()
    def post(t, c):
        return M.postprocess_with_captions(t.long(), [c[:, i] for i in range(c.shape[1])], tok)
    assert post(tok_s, conf_s) == post(tok_ns, conf_ns)
    return firsts


CONTRACT_CASES = [
    ("P", "bf16", 13, {}, 0),
    ("P", "bf16", 37, {"images_per_cluster": 16}, 0),
    ("P", "bf16", 37, {"images_per_cluster": 16}, 5),
    ("P", "bf16", 37, {"images_per_cluster": 8, "ctas_per_sm": 2}, 5),
    ("P", "bf16", 13, {"per_op_kernels": True}, 0),
    ("P", "bf16", 37, {"per_op_kernels": True}, 5),
    ("P", "fp32", 13, {}, 0),
    ("T", "bf16", 16, {}, 0),
]


@pytest.mark.parametrize("config,precision,B,opts,top_k", CONTRACT_CASES)
def test_stop_at_eos_contract(model_p, config, precision, B, opts, top_k):
    model = model_p if config == "P" else _model_t()
    model.set_precision(precision)
    T = 40
    x = cases.images(B, seed=500 + B).to(DEV)
    u = torch.rand(B, T, generator=torch.Generator().manual_seed(B)).to(DEV) if top_k else None
    with M.decode_options(**opts):
        delta = choose_delta(model, x, T)
        with eos_bias(model, delta):
            tn, cn = model.generate_tokens(x, T, top_k=top_k, uniforms=u, use_graph=False)
            ts, cs = model.generate_tokens(x, T, top_k=top_k, uniforms=u, use_graph=False, eos_token=EOS)
            tg, cg = model.generate_tokens(x, T, top_k=top_k, uniforms=u, eos_token=EOS)          # captured graph
    firsts = check_contract(tn, cn, ts, cs, T)
    assert torch.equal(tg, ts) and torch.equal(cg, cs)
    done = [e for e in firsts if e is not None]
    print(f"{config} {precision} B={B} {opts} top_k={top_k}: delta={delta:.3f}, first EOS steps {sorted(done)}, "
          f"{len(firsts) - len(done)} never")
    if top_k == 0:
        assert 0 < len(done) < B and len(set(done)) > 2, firsts


@pytest.mark.parametrize("opts", [{}, {"images_per_cluster": 16}, {"ctas_per_sm": 2}, {"per_op_kernels": True}])
def test_stop_at_eos_extremes(model_p, opts):
    """A huge EOS bias: every image emits EOS at step 0 -> [BOS, EOS, PAD, ...] and confidences [conf_0, 0, ...].  A hugely negative
    one: no image ever emits EOS -> bitwise the no-stop run."""
    model_p.set_precision("bf16")
    B, T = 19, 30
    x = cases.images(B, seed=71).to(DEV)
    with M.decode_options(**opts):
        with eos_bias(model_p, 1e4):
            tn, cn = model_p.generate_tokens(x, T, use_graph=False)
            ts, cs = model_p.generate_tokens(x, T, eos_token=EOS)
        with eos_bias(model_p, -1e4):
            tn2, cn2 = model_p.generate_tokens(x, T, use_graph=False)
            ts2, cs2 = model_p.generate_tokens(x, T, eos_token=EOS)
    want = torch.full((B, T + 1), PAD, dtype=torch.int32, device=DEV)
    want[:, 0], want[:, 1] = BOS, EOS
    assert torch.equal(ts, want), ts[0]
    assert torch.equal(cs[:, 0], cn[:, 0]) and (cs[:, 1:] == 0).all()
    check_contract(tn, cn, ts, cs, T)
    assert torch.equal(ts2, tn2) and torch.equal(cs2, cn2)


@pytest.mark.parametrize("opts", [{}, {"images_per_cluster": 16}, {"per_op_kernels": True}])
def test_stop_at_eos_is_batch_invariant(model_p, opts):
    """An image's result does not depend on which images share its cluster or batch, or on when they finish."""
    model_p.set_precision("bf16")
    T = 40
    x = cases.images(40, seed=81).to(DEV)
    with M.decode_options(**opts):
        delta = choose_delta(model_p, x, T)
        with eos_bias(model_p, delta):
            t40, c40 = model_p.generate_tokens(x, T, eos_token=EOS, use_graph=False)
            t16, c16 = model_p.generate_tokens(x[:16], T, eos_token=EOS, use_graph=False)
            t40b, c40b = model_p.generate_tokens(x, T, eos_token=EOS, use_graph=False)
    assert torch.equal(t40[:16], t16) and torch.equal(c40[:16], c16)
    assert torch.equal(t40, t40b) and torch.equal(c40, c40b)


@pytest.mark.parametrize("opts", [{}, {"per_op_kernels": True}])
def test_stop_at_eos_graph_replays_start_fresh(model_p, opts):
    """Two replays of one captured plan with different images (different EOS patterns) each equal their eager run: no finished state
    leaks from one replay into the next."""
    model_p.set_precision("bf16")
    T, B = 40, 24
    xa, xb = cases.images(B, seed=91).to(DEV), cases.images(B, seed=92).to(DEV)
    with M.decode_options(**opts):
        delta = choose_delta(model_p, xa, T)
        with eos_bias(model_p, delta):
            ga = model_p.generate_tokens(xa, T, eos_token=EOS)
            gb = model_p.generate_tokens(xb, T, eos_token=EOS)
            ga2 = model_p.generate_tokens(xa, T, eos_token=EOS)
            ea = model_p.generate_tokens(xa, T, eos_token=EOS, use_graph=False)
            eb = model_p.generate_tokens(xb, T, eos_token=EOS, use_graph=False)
    assert not torch.equal(ea[0], eb[0])
    for g, e in ((ga, ea), (gb, eb), (ga2, ea)):
        assert torch.equal(g[0], e[0]) and torch.equal(g[1], e[1])


@pytest.mark.parametrize("opts", [{}, {"per_op_kernels": True}])
def test_stop_at_eos_writes_every_skipped_position(model_p, opts):
    """Engine.decode on buffers pre-filled with sentinels: the library writes PAD / 0 itself.  And a decode split in two calls (the
    second starting with some images already finished in its known prefix) equals the single call."""
    model_p.set_precision("bf16")
    T, B = 40, 21
    x = cases.images(B, seed=95).to(DEV)
    with M.decode_options(**opts):
        delta = choose_delta(model_p, x, T)
        with eos_bias(model_p, delta):
            want_t, want_c = model_p.generate_tokens(x, T, eos_token=EOS, use_graph=False)
            eng = model_p._engine()
            _, memory = eng.encode(x, want_enc_out=False, want_memory=True)
            ckv = eng.cross_kv(memory)
            tokens = torch.full((B, T + 1), -7, dtype=torch.int32, device=DEV)
            tokens[:, 0] = BOS
            confs = torch.full((B, (T + 3) // 4), 5.0, dtype=torch.float32, device=DEV)
            eng.decode(ckv, tokens, 0, T, max_tokens=T, forced=False, confs=confs, eos_token=EOS)
            assert torch.equal(tokens, want_t) and torch.equal(confs, want_c)
            k = 17
            tokens2 = torch.full((B, T + 1), -7, dtype=torch.int32, device=DEV)
            tokens2[:, 0] = BOS
            confs2 = torch.full((B, (T + 3) // 4), 5.0, dtype=torch.float32, device=DEV)
            kv, scratch = eng.decode(ckv, tokens2, 0, k, max_tokens=T, forced=False, confs=confs2, eos_token=EOS)
            eng.decode(ckv, tokens2, k, T, max_tokens=T, forced=False, confs=confs2, eos_token=EOS, kv=kv, scratch=scratch)
    finished_early = ((want_t[:, 1:k + 1] == EOS).any(1)).sum().item()
    assert 0 < finished_early < B
    assert torch.equal(tokens2, want_t) and torch.equal(confs2, want_c)


def test_stop_at_eos_through_the_pipeline(model_p):
    """generate_stream(..., stop_at_eos=True) and a GenerationPipeline with top-k sampling equal the serial stop runs, including a
    ragged last batch."""
    model_p.set_precision("bf16")
    tok = M.Tokenizer()
    T = 40
    xs = [cases.images(16, seed=600 + i) for i in range(4)] + [cases.images(5, seed=700)]
    delta = choose_delta(model_p, xs[0].to(DEV), T)
    with eos_bias(model_p, delta):
        want = [M.generate(model_p, x.to(DEV), tok, max_len=T, stop_at_eos=True) for x in xs]
        nostop = [M.generate(model_p, x.to(DEV), tok, max_len=T) for x in xs]
        got = list(M.generate_stream(model_p, (x.pin_memory() for x in xs), tok, max_len=T, stop_at_eos=True))
        pipe = M.GenerationPipeline(model_p, 16, T, top_k=5, depth=3, decode_streams=2, eos_token=EOS)
        us = [torch.rand(16, T, generator=torch.Generator().manual_seed(i)).to(DEV) for i in range(4)]
        tickets = [pipe.submit(xs[i].to(DEV), uniforms=us[i]) for i in range(4)]
        pipe.join()
        refs = [model_p.generate_tokens(xs[i].to(DEV), T, top_k=5, uniforms=us[i], eos_token=EOS) for i in range(4)]
    assert len(got) == len(want)
    for (gt, gc), (wt, wc), (nt, nc) in zip(got, want, nostop):
        assert torch.equal(gt, wt) and len(gc) == len(wc) and all(torch.equal(a, b) for a, b in zip(gc, wc))
        check_contract(nt, torch.stack(nc, 1), wt, torch.stack(wc, 1), T)
    for t, (rt, rc) in zip(tickets, refs):
        ht, hc = t.result()
        assert torch.equal(ht, rt) and torch.equal(hc, rc)


def _replay_ms(model, x, T, reps=5, **kw):
    for _ in range(2):
        model.generate_tokens(x, T, **kw)
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); model.generate_tokens(x, T, **kw); b.record(); torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[reps // 2]


@pytest.mark.parametrize("config,B,bound", [("P", 64, 0.5), ("T", 16, 0.6)])
def test_stop_at_eos_actually_stops(model_p, config, B, bound):
    """Every image finishing at step 0: the graph-replayed call is far cheaper than the full T = 99 steps -- the fused kernel leaves its
    step loop, the per-operation chain's launches return at entry."""
    model = model_p if config == "P" else _model_t()
    model.set_precision("bf16")
    x = cases.images(B, seed=31).to(DEV)
    with eos_bias(model, 1e4):
        full = _replay_ms(model, x, 99)
        stop = _replay_ms(model, x, 99, eos_token=EOS)
    print(f"config {config} B={B} T=99, every image at EOS from step 0: {full:.2f} ms without stopping, {stop:.2f} ms with "
          f"({stop / full:.2f}x)")
    assert stop < bound * full


def test_stop_at_eos_rejected_arguments(model_p):
    model_p.set_precision("bf16")
    x = cases.images(3, seed=5).to(DEV)
    with pytest.raises(ValueError):
        model_p.generate_tokens(x, 10, return_logits=True, eos_token=EOS)
    with pytest.raises(ValueError):
        model_p.generate_tokens(x, 10, eos_token=305)
    with pytest.raises(ValueError):
        model_p.generate_tokens(x, 10, eos_token=-1)
    eng = model_p._engine()
    _, memory = eng.encode(x, want_enc_out=False, want_memory=True)
    ckv = eng.cross_kv(memory)
    tokens = torch.full((3, 11), PAD, dtype=torch.int32, device=DEV)
    tokens[:, 0] = BOS
    with pytest.raises(M._lib.MdcError):                       # teacher forcing + stop
        eng.decode(ckv, tokens, 0, 10, max_tokens=10, forced=True, eos_token=EOS)
    with pytest.raises(M._lib.MdcError):                       # out of range at the C ABI
        eng.decode(ckv, tokens, 0, 10, max_tokens=10, forced=False, eos_token=305)
    class BadPad(M.Tokenizer):
        PAD_code = 0
    with pytest.raises(ValueError):
        M.generate(model_p, x, BadPad(), max_len=10, stop_at_eos=True)
