"""GPU: prompted beam search (generate_beam_tokens(..., prompt=, prompt_lengths=), generate_beam(..., prompt=), mdc_beam_state.prompt_len).

1. Every length 0 is bitwise the unprompted search.  2. fp32 ragged prompts against the prompted beam oracle (tests/prompt_beam_oracle.py).
3. One beam is prompted greedy generate_tokens, prefilled and step by step, on the fused kernel (config P) and on the per-operation chain
(config T).  4. K = 4: the all-positions prefill against the step path.  5. Graph replay, batch invariance and a cached plan reused with
another prompt.  6. Rejections before any launch.  7. A caption prompt comes back from postprocess_with_captions."""
import pytest
import torch

pytestmark = pytest.mark.gpu

import mdcnet_b200 as M  # noqa: E402
from mdcnet_b200.model import BeamPlan  # noqa: E402
from oracle import cases  # noqa: E402
from tests.eos_helpers import EOS, eos_bias  # noqa: E402
from tests.prompt_beam_oracle import generate_beam  # noqa: E402

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


def _prompts(B, P, lens, seed):
    """Caption-like prompts [SOC, words...] of the given lengths (words from 270 up, PAD past each length)."""
    g = torch.Generator().manual_seed(seed)
    prompt = torch.randint(270, 299, (B, P), generator=g)
    prompt[:, 0] = SOC
    lens = torch.as_tensor(lens).long()
    prompt[torch.arange(P)[None, :] >= lens[:, None]] = PAD
    return prompt, lens


def _beam_plans(model, B, T, K):
    """The cached beam plans of one (B, T, K) shape."""
    return [p for k, p in model.__dict__.get("_plans", {}).items()
            if k != "eng" and isinstance(p, BeamPlan) and (p.B, p.T, p.K) == (B, T, K)]


def _selection_margins(logits, lens, K, T):
    """Per image, the smallest gap between the K-th and (K+1)-th candidate over its free steps, replaying the beam selection in f32 on a
    search's own step logits (BeamPlan.logits: row r's step-t logits in row order after step t-1's reorder)."""
    B, V = lens.shape[0], logits.shape[-1]
    score = torch.full((B, K), -float("inf"), device=DEV)
    score[:, 0] = 0
    fin = torch.full((B, K), -1, dtype=torch.long, device=DEV)
    margin = torch.full((B,), float("inf"), dtype=torch.float64, device=DEV)
    lens = lens.to(DEV)
    for t in range(T):
        lg = logits[:, t].view(B, K, V)
        m = lg.max(-1, keepdim=True).values
        lp = (lg - m) - torch.log(torch.exp(lg - m).sum(-1, keepdim=True))
        cand = score[..., None] + lp
        done = fin >= 0
        cand[done] = -float("inf")
        cand[..., PAD] = torch.where(done, score, cand[..., PAD])
        top, idx = cand.view(B, K * V).topk(K + 1, dim=-1)
        gap = (top[:, K - 1].double() - top[:, K].double()).nan_to_num(float("inf"))
        free = t >= lens
        margin = torch.where(free, torch.minimum(margin, gap), margin)
        parent, tok = idx[:, :K] // V, idx[:, :K] % V
        pf = fin.gather(1, parent)
        new_fin = torch.where(pf >= 0, pf, torch.where(tok == EOS, torch.full_like(tok, t), torch.full_like(tok, -1)))
        score = torch.where(free[:, None], top[:, :K], score)
        fin = torch.where(free[:, None], new_fin, fin)
    return margin.cpu()


# ---- 1. every length 0 is the unprompted search --------------------------------------------------------------------------------
@pytest.mark.parametrize("precision,opts", [("bf16", {}), ("bf16", {"per_op_kernels": True}), ("fp32", {})])
def test_zero_lengths_are_bitwise_unprompted(model_p, precision, opts):
    model_p.set_precision(precision)
    B, K, T = 6, 4, 24
    x = cases.images(B, seed=201).to(DEV)
    with M.decode_options(**opts):
        want = model_p.generate_beam_tokens(x, T, K, eos_token=EOS)
        got = model_p.generate_beam_tokens(x, T, K, eos_token=EOS, prompt=torch.full((B, 5), 280), prompt_lengths=[0] * B)
    for a, b in zip(got, want):
        assert torch.equal(a, b)


# ---- 2. fp32: ragged prompts against the oracle (the step path: the prefill does not cover fp32) ------------------------------------
SEEDS = [1000, 1001, 1002, 1003, 1004, 1005, 1006, 1007]
MARGIN = 1e-4


def test_fp32_ragged_prompts_equal_the_oracle(model_p):
    sd, cfg = cases.state_dict_of(model_p.cpu()), cases.oracle_cfg("P")
    model_p.to(DEV).set_precision("fp32")
    K, T = 3, 20
    for seed in SEEDS:
        x = cases.images(4, seed=seed)
        prompt, lens = _prompts(4, 12, [0, 3, 7, 12], seed)
        want_t, want_s, want_l, margin, want_c = generate_beam(sd, x, cfg, T, K, prompt=prompt, lengths=lens, return_confs=True)
        if margin > MARGIN:
            break
    else:
        pytest.fail(f"no seed of {SEEDS} keeps the oracle's selection margins above {MARGIN}")
    tok, norm, lp, conf = model_p.generate_beam_tokens(x.to(DEV), T, K, eos_token=EOS, prompt=prompt, prompt_lengths=lens)
    assert torch.equal(tok.cpu().long(), want_t), (seed, margin)
    assert (lp.cpu() - want_l).abs().max().item() <= 1e-4
    assert (norm.cpu() - want_s).abs().max().item() <= 1e-4
    assert (conf.cpu() - want_c).abs().max().item() <= 1e-4
    for b, l in enumerate(lens.tolist()):
        assert (lp[b, :, :l] == 0).all()


# ---- 3. one beam is prompted greedy -------------------------------------------------------------------------------------------
def _one_beam_is_greedy(model, x, T, prompt, lens, prefill):
    with M.decode_options(prefill=prefill):
        _, _, lg = model.generate_tokens(x, T, prompt=prompt, prompt_lengths=lens, return_logits=True, use_graph=False)
        want, want_c = model.generate_tokens(x, T, prompt=prompt, prompt_lengths=lens, eos_token=EOS)     # a beam ends at EOS too
        tok, norm, lp, conf = model.generate_beam_tokens(x, T, 1, eos_token=EOS, prompt=prompt, prompt_lengths=lens)
    n = int(lens.min())
    assert any(p.prefill == (n if prefill else 0) for p in _beam_plans(model, x.shape[0], T, 1))
    top2 = lg.topk(2, dim=-1).values
    margin = (top2[..., 0] - top2[..., 1]).cpu()
    tok, want = tok[:, 0].cpu(), want.cpu()
    conf, want_c = conf[:, 0].cpu(), want_c.cpu()
    compared = 0
    for b in range(x.shape[0]):
        l = int(lens[b])
        assert torch.equal(tok[b, 1:1 + l], prompt[b, :l].int())
        diff = (tok[b] != want[b]).nonzero()
        d = int(diff[0]) - 1 if len(diff) else T          # the step that chose the first differing token
        if d < T:                                          # only where log-softmax rounding can turn a near-tie around
            assert margin[b, d].item() <= 1e-4, (b, d, margin[b, d].item())
        else:
            compared += 1
        assert (conf[b, :(d + 3) // 4] - want_c[b, :(d + 3) // 4]).abs().max().item() <= 1e-5
    assert compared >= x.shape[0] - 1


@pytest.mark.parametrize("prefill", [True, False])
def test_bf16_one_beam_is_prompted_greedy(model_p, prefill):
    model_p.set_precision("bf16")
    B, T = 16, 60
    x = cases.images(B, seed=211).to(DEV)
    prompt, lens = _prompts(B, 14, torch.randint(6, 15, (B,), generator=torch.Generator().manual_seed(3)), 211)
    _one_beam_is_greedy(model_p, x, T, prompt, lens, prefill)


def test_config_t_one_beam_is_prompted_greedy_and_prefills(model_t):
    model_t.set_precision("bf16")
    B, T = 4, 24
    x = cases.images(B, seed=221).to(DEV)
    prompt, lens = _prompts(B, 9, [6, 9, 7, 8], 221)
    eng = model_t._engine()
    assert eng.lib.mdc_decode_prefill_workspace_bytes(eng.handle, B, 6) > 0
    _one_beam_is_greedy(model_t, x, T, prompt, lens, True)
    with M.decode_options(prefill=True):
        tok, norm, lp, conf = model_t.generate_beam_tokens(x, T, 4, eos_token=EOS, prompt=prompt, prompt_lengths=lens)
    assert any(p.prefill == 6 for p in _beam_plans(model_t, B, T, 4))
    for b, l in enumerate(lens.tolist()):
        assert (tok[b, :, 1:1 + l].cpu() == prompt[b, :l]).all() and (lp[b, :, :l] == 0).all()
        assert (lp[b, :, l] < 0).all() and torch.isfinite(norm[b]).all()


# ---- 4. K = 4: the prefill against the step path --------------------------------------------------------------------------------
def test_bf16_prefill_matches_the_step_path(model_p):
    model_p.set_precision("bf16")
    B, K, T = 16, 4, 40
    x = cases.images(B, seed=231).to(DEV)
    prompt, lens = _prompts(B, 16, torch.randint(6, 17, (B,), generator=torch.Generator().manual_seed(4)), 231)
    n = int(lens.min())
    runs = {}
    for prefill in (False, True):
        with M.decode_options(prefill=prefill):
            runs[prefill] = model_p.generate_beam_tokens(x, T, K, eos_token=EOS, prompt=prompt, prompt_lengths=lens)
            plan = next(p for p in _beam_plans(model_p, B, T, K) if p.prefill == (n if prefill else 0))
            if not prefill:
                step_logits = plan.logits.clone()
    margin = _selection_margins(step_logits, lens, K, T)
    tok_s, norm_s, lp_s, conf_s = (o.cpu() for o in runs[False])
    tok_p, norm_p, lp_p, conf_p = (o.cpu() for o in runs[True])
    gaps = (norm_s[:, :-1] - norm_s[:, 1:]).min(-1).values.double()      # the final ordering's margin
    margin = torch.minimum(margin, gaps)
    compared = 0
    for b, l in enumerate(lens.tolist()):
        cols = [t // 4 for t in range(0, l, 4)]
        assert (conf_s[b][:, cols] - conf_p[b][:, cols]).abs().max().item() <= BOUND      # prompt-step confidences
        assert (tok_p[b, :, 1:1 + l] == prompt[b, :l]).all() and (lp_p[b, :, :l] == 0).all()
        if margin[b] > BOUND:
            assert torch.equal(tok_s[b], tok_p[b]), (b, margin[b].item())
        if torch.equal(tok_s[b], tok_p[b]):
            compared += 1
            assert (lp_s[b] - lp_p[b]).abs().max().item() <= BOUND
            assert (norm_s[b] - norm_p[b]).abs().max().item() <= BOUND
    print(f"prefill vs step path: {compared} of {B} images with equal beams; selection margins {margin.tolist()}")
    assert compared >= B // 2


# ---- 5. graph replay, batch invariance, a cached plan with another prompt ------------------------------------------------------
@pytest.mark.parametrize("prefill", [False, True])
def test_graph_replay_batch_invariance_and_plan_reuse(model_p, prefill):
    model_p.set_precision("bf16")
    B, K, T, P = 16, 4, 30, 12
    x = cases.images(B, seed=241).to(DEV)
    p1, l1 = _prompts(B, P, torch.randint(6, P + 1, (B,), generator=torch.Generator().manual_seed(5)), 1)
    p2, l2 = _prompts(B, P, torch.randint(6, P + 1, (B,), generator=torch.Generator().manual_seed(6)), 2)
    l1[0] = l2[0] = 6                                     # the same min(l_b): one plan for both prompts
    with M.decode_options(prefill=prefill):
        g1 = model_p.generate_beam_tokens(x, T, K, eos_token=EOS, prompt=p1, prompt_lengths=l1)
        e1 = model_p.generate_beam_tokens(x, T, K, eos_token=EOS, prompt=p1, prompt_lengths=l1, use_graph=False)
        g2 = model_p.generate_beam_tokens(x, T, K, eos_token=EOS, prompt=p2, prompt_lengths=l2)      # the cached plan
        again = model_p.generate_beam_tokens(x, T, K, eos_token=EOS, prompt=p2, prompt_lengths=l2)
        model_p.__dict__["_plans"].clear()
        fresh = model_p.generate_beam_tokens(x, T, K, eos_token=EOS, prompt=p2, prompt_lengths=l2)
        x40 = torch.cat([cases.images(24, seed=242).to(DEV), x])
        p40, l40 = torch.cat([_prompts(24, P, [6] * 24, 3)[0], p2]), torch.cat([torch.full((24,), 6), l2])
        all40 = model_p.generate_beam_tokens(x40, T, K, eos_token=EOS, prompt=p40, prompt_lengths=l40)
    assert any(p.prefill == (6 if prefill else 0) for p in _beam_plans(model_p, 40, T, K))
    for a, b, c, d, e, f in zip(g1, e1, g2, again, fresh, all40):
        assert torch.equal(a, b) and torch.equal(c, d) and torch.equal(c, e) and torch.equal(c, f[24:])
    assert not torch.equal(g1[0], g2[0])


# ---- 6. rejections before any launch -------------------------------------------------------------------------------------------
def test_rejections_before_any_launch(model_p):
    model_p.set_precision("bf16")
    x = cases.images(2, seed=5).to(DEV)
    T = 10
    tokz = M.Tokenizer()
    model_p._engine()
    ok = torch.tensor([[SOC, 280, EOC], [SOC, 281, EOC]])
    bad = [
        dict(prompt=torch.tensor([[SOC, PAD, EOC], [SOC, 281, EOC]])),
        dict(prompt=torch.tensor([[SOC, EOS, EOC], [SOC, 281, EOC]])),
        dict(prompt=ok, prompt_lengths=[4, 3]),
        dict(prompt=ok, prompt_lengths=[-1, 3]),
        dict(prompt=torch.tensor([[SOC, 400, EOC], [SOC, 281, EOC]])),
        dict(prompt=ok[:1]),
        dict(prompt=ok.float()),
        dict(prompt_lengths=[1, 1]),
    ]
    torch.cuda.synchronize()
    n0 = L.launch_count(DEV)
    for kw in bad:
        with pytest.raises(ValueError):
            model_p.generate_beam_tokens(x, T, 2, eos_token=EOS, **kw)
        with pytest.raises(ValueError):
            M.generate_beam(model_p, x, tokz, max_len=T, num_beams=2, **kw)
    for TT in (3, 2):                                      # l_b = 3 = T and l_b > T: no step left to search
        with pytest.raises(ValueError):
            model_p.generate_beam_tokens(x, TT, 2, eos_token=EOS, prompt=ok)
        with pytest.raises(ValueError):
            M.generate_beam(model_p, x, tokz, max_len=TT, num_beams=2, prompt=ok)
    assert L.launch_count(DEV) == n0
    model_p.generate_beam_tokens(x, 4, 2, eos_token=EOS, prompt=ok)       # l_b = T - 1 is accepted
    assert L.launch_count(DEV) > n0


# ---- 7. a caption prompt comes back from postprocess_with_captions --------------------------------------------------------------
def test_caption_prompt_roundtrip(model_p):
    """A huge EOS bias makes EOS the best continuation at every free step: each image's best beam keeps its caption and ends right
    after it, at column 6, which the reference's (EOS - 1) % 5 rule accepts."""
    model_p.set_precision("bf16")
    words = {280: "crack", 281: "patch", 282: "scratch", 283: "inclusion"}
    tok = M.Tokenizer(vocab=words)
    prompt, lens = tok.caption_prompt([[280, 281, 282], [283, 280, 280]])
    x = cases.images(2, seed=81).to(DEV)
    with eos_bias(model_p, 1e4):
        seqs, confs = M.generate_beam(model_p, x, tok, max_len=12, num_beams=4, prompt=prompt, prompt_lengths=lens)
    assert seqs[:, 1:6].tolist() == prompt.tolist() and (seqs[:, 6] == EOS).all() and (seqs[:, 7:] == PAD).all()
    _, _, captions, _ = M.postprocess_with_captions(seqs, confs, tok)
    assert captions == [["crack", "patch", "scratch"], ["inclusion", "crack", "crack"]]
