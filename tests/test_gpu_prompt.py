"""GPU: prompted generation (generate(..., prompt=, prompt_lengths=), generate_tokens(..., prompt=), mdc_decode_state.prompt_len,
mdc_decode_prefill_steps).

1. With a prompt equal to the row's own unprompted output (ragged, including 0 and T), the step path is bitwise the unprompted run.
2. Foreign prompts: fp32 tokens equal the prompted oracle, bf16 logits stay within the 2e-2 contract, free tokens are the argmax of
   their own logits, and the prompt columns are kept (also when stopping at EOS).
3. The all-positions prefill of a prompt against the step path: KV pages, logits, tokens and prompt-step confidences.
4. Graph replay and batch invariance.  5. Rejected arguments.  6. A caption prompt comes back from postprocess_with_captions."""

import pytest
import torch

pytestmark = pytest.mark.gpu

import mdcnet_b200 as M  # noqa: E402
from oracle import cases, mdc_oracle as O  # noqa: E402
from tests.eos_helpers import EOS, eos_bias  # noqa: E402
from tests.gpu_util import cos  # noqa: E402
from tests.prompt_oracle import generate_prompted  # noqa: E402

L = M._lib
DEV = "cuda"
PAD, BOS, SOC, EOC = 302, 300, 303, 304
BOUND = 1.5e-2          # the prefill-vs-autoregressive logit bound of the all-positions pass (tests/test_gpu_model.py)


@pytest.fixture(scope="module")
def model_p():
    return cases.build_product_model("P", seed=0, gamma_seed=5).to(DEV)


@pytest.fixture(scope="module")
def model_t():
    return cases.build_product_model("T", seed=0, gamma_seed=5).to(DEV)


def _own_prompts(tok, lengths):
    """Each row's own unprompted output as its prompt, cut before its first PAD or EOS (neither may be a prompt token)."""
    new = tok[:, 1:].cpu().long()
    cut = []
    for b, l in enumerate(lengths):
        bad = ((new[b] == PAD) | (new[b] == EOS)).nonzero()
        cut.append(min(l, int(bad[0]) if len(bad) else l))
    return new, torch.tensor(cut)


def _caption_prompts(B, P, seed):
    """Caption-like prompts [SOC, words..., EOC] of ragged lengths 0..P (words from 270 up)."""
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(0, P + 1, (B,), generator=g)
    lens[0], lens[-1] = 0, P
    prompt = torch.full((B, P), PAD, dtype=torch.long)
    for b, l in enumerate(lens.tolist()):
        if l:
            prompt[b, :l] = torch.randint(270, 299, (l,), generator=g)
            prompt[b, 0] = SOC
            if l > 1:
                prompt[b, l - 1] = EOC
    return prompt, lens


# ---- 1. bitwise equality with the unprompted run -------------------------------------------------------------------------------
BITWISE_CASES = [
    ("P", "bf16", {}), ("P", "bf16", {"images_per_cluster": 16}), ("P", "bf16", {"ctas_per_sm": 2}),
    ("P", "bf16", {"per_op_kernels": True}), ("P", "fp32", {}), ("T", "bf16", {}),
]


@pytest.mark.parametrize("config,precision,opts", BITWISE_CASES)
@pytest.mark.parametrize("top_k", [0, 5])
@pytest.mark.parametrize("eos", [None, EOS])
def test_own_prompt_is_bitwise_unprompted(request, config, precision, opts, top_k, eos):
    model = request.getfixturevalue("model_p" if config == "P" else "model_t")
    model.set_precision(precision)
    B, T = 13, 24
    x = cases.images(B, seed=300 + B).to(DEV)
    u = torch.rand(B, T, generator=torch.Generator().manual_seed(7)).to(DEV)
    lengths = [0, T, 1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 23]
    with M.decode_options(prefill=False, **opts):
        want_t, want_c = model.generate_tokens(x, T, top_k=top_k, uniforms=u, use_graph=False, eos_token=eos)
        prompt, lens = _own_prompts(want_t, lengths)
        got_t, got_c = model.generate_tokens(x, T, top_k=top_k, uniforms=u, use_graph=False, eos_token=eos, prompt=prompt,
                                             prompt_lengths=lens)
    assert torch.equal(got_t, want_t)
    assert torch.equal(got_c, want_c)


# ---- 2. foreign prompts ---------------------------------------------------------------------------------------------------------
def test_fp32_foreign_prompt_equals_the_oracle(model_p):
    sd, cfg = cases.state_dict_of(model_p.cpu()), cases.oracle_cfg("P")
    model_p.to(DEV).set_precision("fp32")
    B, T, P = 4, 20, 9
    for seed in range(40, 48):            # the first seed whose oracle run has no near-tie at a free step
        x = cases.images(B, seed=seed)
        prompt, lens = _caption_prompts(B, P, seed)
        want_t, _, lg = generate_prompted(sd, x, cfg, T, prompt, lens, return_logits=True)
        top2 = lg.topk(2, -1).values
        free = torch.arange(T)[None, :] >= lens[:, None]
        if ((top2[..., 0] - top2[..., 1])[free]).min().item() > 1e-4:
            break
    else:
        pytest.fail("no seed without a near-tie")
    got, _ = model_p.generate_tokens(x.to(DEV), T, prompt=prompt, prompt_lengths=lens)
    assert torch.equal(got.cpu().long(), want_t)


@pytest.mark.parametrize("opts", [{}, {"per_op_kernels": True}])
def test_bf16_foreign_prompt_logits(model_p, opts):
    sd, cfg = cases.state_dict_of(model_p.cpu()), cases.oracle_cfg("P")
    model_p.to(DEV).set_precision("bf16")
    B, T, P = 16, 40, 14
    x = cases.images(B, seed=55)
    prompt, lens = _caption_prompts(B, P, 55)
    with M.decode_options(**opts):
        tok, conf, lg = model_p.generate_tokens(x.to(DEV), T, prompt=prompt, prompt_lengths=lens, return_logits=True)
        tok_s, _ = model_p.generate_tokens(x.to(DEV), T, prompt=prompt, prompt_lengths=lens, eos_token=EOS)
    tok, lg, tok_s = tok.cpu().long(), lg.cpu(), tok_s.cpu().long()
    for b in range(B):
        l = int(lens[b])
        assert torch.equal(tok[b, 1:1 + l], prompt[b, :l]) and torch.equal(tok_s[b, 1:1 + l], prompt[b, :l])
        free = lg[b, l:].argmax(-1)
        assert torch.equal(tok[b, 1 + l:], free), b
    seqs = tok[:, :T]
    with torch.no_grad():
        enc = O.encoder_forward(sd, x, cfg)
        h = sd["decoder.embedding.weight"][seqs] + sd["decoder.decoder_pos_embed"][:, :T]
        y = O.decoder_stack(sd, h, enc + sd["decoder.encoder_pos_embed"], seqs, cfg)
        want = y @ sd["decoder.output.weight"].T + sd["decoder.output.bias"]
    err = (lg - want).abs().max().item()
    print(f"bf16 prompted logits {opts}: max|d| = {err:.3e}, cos = {cos(lg, want):.6f}")
    assert err <= 2e-2 and cos(lg, want) >= 0.999


# ---- 3. the prefill path against the step path ----------------------------------------------------------------------------------
def _engine_run(model, x, tokens, lens, T, n_end, prefill):
    """Steps [0, n_end) of a prompted decode through Engine.decode, on fresh buffers: (tokens, kv, logits, confs)."""
    eng = model._engine()
    _, memory = eng.encode(x, want_enc_out=False, want_memory=True)
    ckv = eng.cross_kv(memory)
    B = x.shape[0]
    tokens = tokens.clone()
    logits = torch.zeros((B, T, eng.dims.vocab), dtype=torch.float32, device=DEV)
    confs = torch.zeros((B, (T + 3) // 4), dtype=torch.float32, device=DEV)
    ws = None
    if prefill:
        ws = torch.empty(eng.lib.mdc_decode_prefill_workspace_bytes(eng.handle, B, prefill), dtype=torch.uint8, device=DEV)
    kv, _ = eng.decode(ckv, tokens, 0, n_end, max_tokens=T, forced=False, logits=logits, confs=confs,
                       prompt_len=lens.to(DEV, torch.int32), prefill=prefill, prefill_ws=ws)
    return tokens, kv, logits, confs


@pytest.mark.parametrize("config", ["P", "T"])
def test_prefill_matches_the_step_path(request, config):
    model = request.getfixturevalue("model_p" if config == "P" else "model_t")
    model.set_precision("bf16")
    B, T, P = 24, 32, 18
    x = cases.images(B, seed=61).to(DEV)
    prompt, lens = _caption_prompts(B, P, 61)
    lens = lens.clamp(min=5)                     # min(l_b) >= 1: the prefill covers the first 5 steps of every row
    for b, l in enumerate(lens.tolist()):
        prompt[b, :l] = torch.where(prompt[b, :l] == PAD, torch.full_like(prompt[b, :l], 280), prompt[b, :l])
    n = int(lens.min())
    tokens = torch.full((B, T + 1), PAD, dtype=torch.int32, device=DEV)
    tokens[:, 0] = BOS
    tokens[:, 1:1 + P] = torch.where(torch.arange(P)[None, :] < lens[:, None], prompt, torch.full_like(prompt, PAD)).to(DEV, torch.int32)
    eng = model._engine()
    assert eng.lib.mdc_decode_prefill_workspace_bytes(eng.handle, B, n) > 0
    # KV positions 0..n-1 after the first n steps
    _, kv_s, _, _ = _engine_run(model, x, tokens, lens, T, n, 0)
    _, kv_p, _, _ = _engine_run(model, x, tokens, lens, T, n, n)
    assert torch.equal(kv_s.page_table, kv_p.page_table)
    a, b = kv_s.pool.float(), kv_p.pool.float()
    kv_err, kv_scale = (a - b).abs().max().item(), a.abs().max().item()
    print(f"{config}: KV of the {n} prefilled positions max|d| = {kv_err:.3e} (max|K,V| = {kv_scale:.3f}), cos = {cos(a, b):.6f}")
    assert kv_err <= 2e-2 * max(1.0, kv_scale) and cos(a, b) >= 0.9999
    # the whole call
    tok_s, _, lg_s, cf_s = _engine_run(model, x, tokens, lens, T, T, 0)
    tok_p, _, lg_p, cf_p = _engine_run(model, x, tokens, lens, T, T, n)
    top2 = lg_s.topk(2, -1).values
    margin = (top2[..., 0] - top2[..., 1]).cpu()
    worst = 0.0
    for r in range(B):
        diff = (tok_s[r, 1:] != tok_p[r, 1:]).nonzero()
        d = int(diff[0]) if len(diff) else T          # first differing token column - 1 = the step that chose it
        if d < T:
            assert margin[r, d].item() <= BOUND, (r, d, margin[r, d].item())
        worst = max(worst, (lg_s[r, :d + 1 if d < T else T] - lg_p[r, :d + 1 if d < T else T]).abs().max().item())
        steps = [t for t in range(0, int(lens[r]), 4)]
        assert (cf_s[r, [t // 4 for t in steps]] - cf_p[r, [t // 4 for t in steps]]).abs().max().item() <= BOUND
    print(f"{config}: prefill vs step logits max|d| = {worst:.3e}")
    assert worst <= BOUND


# ---- 4. graph replay and batch invariance ------------------------------------------------------------------------------------
@pytest.mark.parametrize("prefill", [False, True])
def test_graph_replay_and_batch_invariance(model_p, prefill):
    model_p.set_precision("bf16")
    T, P = 30, 12
    with M.decode_options(prefill=prefill):
        x = cases.images(16, seed=71).to(DEV)
        p1, l1 = _caption_prompts(16, P, 1)
        p2, l2 = _caption_prompts(16, P, 2)
        l1, l2 = l1.clamp(min=6), l2.clamp(min=6)          # the same min(l_b): one plan for both prompts
        p1[p1 == PAD], p2[p2 == PAD] = 280, 281
        for p, l in ((p1, l1), (p2, l2)):
            tg, cg = model_p.generate_tokens(x, T, prompt=p, prompt_lengths=l)
            te, ce = model_p.generate_tokens(x, T, prompt=p, prompt_lengths=l, use_graph=False)
            assert torch.equal(tg, te) and torch.equal(cg, ce)
        x40 = torch.cat([cases.images(24, seed=72).to(DEV), x])
        p40, l40 = torch.cat([torch.full((24, P), 282), p2]), torch.cat([torch.full((24,), 6), l2])
        t40, c40 = model_p.generate_tokens(x40, T, prompt=p40, prompt_lengths=l40)
    assert torch.equal(t40[24:], tg) and torch.equal(c40[24:], cg)


# ---- 5. rejections -------------------------------------------------------------------------------------------------------------
def test_rejections(model_p):
    model_p.set_precision("bf16")
    x = cases.images(2, seed=5).to(DEV)
    T = 10
    ok = torch.tensor([[SOC, 280, EOC], [SOC, 281, EOC]])
    bad = [
        dict(prompt=torch.tensor([[SOC, PAD, EOC], [SOC, 281, EOC]])),
        dict(prompt=torch.tensor([[SOC, EOS, EOC], [SOC, 281, EOC]])),
        dict(prompt=ok, prompt_lengths=[4, 3]),
        dict(prompt=ok, prompt_lengths=[-1, 3]),
        dict(prompt=torch.tensor([[SOC, 400, EOC], [SOC, 281, EOC]])),
        dict(prompt=ok[:1]),
        dict(prompt_lengths=[1, 1]),
    ]
    for kw in bad:
        with pytest.raises(ValueError):
            model_p.generate_tokens(x, T, **kw)
    with pytest.raises(ValueError):
        model_p.generate_tokens(x, 2, prompt=ok)                  # l_b = 3 > T = 2
    with pytest.raises(ValueError):
        M.generate(model_p, x, M.Tokenizer(), max_len=2, prompt=ok)
    eng = model_p._engine()
    _, memory = eng.encode(x, want_enc_out=False, want_memory=True)
    tokens = torch.full((2, T + 1), PAD, dtype=torch.int32, device=DEV)
    with pytest.raises(L.MdcError):
        eng.decode(eng.cross_kv(memory), tokens, 0, T, max_tokens=T, forced=True,
                   logits=torch.empty((2, T, eng.dims.vocab), device=DEV), prompt_len=torch.ones(2, dtype=torch.int32, device=DEV))


# ---- 6. a caption prompt comes back from postprocess_with_captions ---------------------------------------------------------------
def test_caption_prompt_roundtrip(model_p):
    """A huge EOS bias makes every free step pick EOS: the prompt steps must still keep the caption (a prompt step never counts as
    EOS), and the step after it ends the sequence at column 6, which the reference's (EOS - 1) % 5 rule accepts."""
    model_p.set_precision("bf16")
    words = {280: "crack", 281: "patch", 282: "scratch", 283: "inclusion"}
    tok = M.Tokenizer(vocab=words)
    prompt, lens = tok.caption_prompt([[280, 281, 282], [283, 280, 280]])
    x = cases.images(2, seed=81).to(DEV)
    with eos_bias(model_p, 1e4):
        seqs, confs = M.generate(model_p, x, tok, max_len=12, prompt=prompt, prompt_lengths=lens, stop_at_eos=True)
    assert seqs[:, 1:6].tolist() == prompt.tolist() and (seqs[:, 6] == EOS).all() and (seqs[:, 7:] == PAD).all()
    _, _, captions, _ = M.postprocess_with_captions(seqs, confs, tok)
    assert captions == [["crack", "patch", "scratch"], ["inclusion", "crack", "crack"]]
