"""GPU: beam search (EncoderDecoder.generate_beam_tokens, generate_beam, mdc_beam_step / mdc_beam_finalize).

Beam search runs T teacher-forced one-step decode windows over the B*K rows, with the beam bookkeeping between them.  The first test
checks that premise: one-step windows give the same logits, bit for bit, as one teacher-forced call.  The rest compare against the
oracle's beam search (fp32), against greedy generate_tokens (K = 1, bf16), against a teacher-forced rescoring of every returned beam
(which needs no KV reorder), and check the EOS / length-penalty contract with EOS raised to arrive at spread-out steps (the eos_bias /
choose_delta technique of the stop-at-EOS tests)."""
import contextlib
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

import mdcnet_b200 as M  # noqa: E402
from oracle import cases, mdc_oracle as O  # noqa: E402
from tests.beam_oracle import generate_beam  # noqa: E402

L = M._lib
DEV = "cuda"
EOS, PAD, BOS = 301, 302, 300


@pytest.fixture(scope="module")
def model_p():
    return cases.build_product_model("P", seed=0, gamma_seed=5).to(DEV)


@pytest.fixture(scope="module")
def model_s():
    return cases.build_product_model("S", seed=0, gamma_seed=5).to(DEV)


@pytest.fixture(scope="module")
def model_t():
    return cases.build_product_model("T", seed=0, gamma_seed=5).to(DEV)


@contextlib.contextmanager
def eos_bias(model, delta):
    b = model.decoder.output.bias
    with torch.no_grad():
        saved = b[EOS].clone()
        b[EOS] += delta
    try:
        yield model
    finally:
        with torch.no_grad():
            b[EOS] = saved


def choose_delta(model, x, T, **kw):
    """delta for which some but not all images emit EOS within T steps (greedy), at as many different steps as possible, with no
    margin within 1e-3 of delta."""
    _, _, lg = model.generate_tokens(x, T, return_logits=True, use_graph=False, **kw)
    others = lg.clone()
    others[..., EOS] = -float("inf")
    margin = (others.max(-1).values - lg[..., EOS]).double().cpu()          # (B, T)
    vals = margin.flatten().unique()                                          # sorted
    mids = (vals[:-1] + vals[1:]) / 2
    cands = mids[(vals[1:] - vals[:-1]) > 2e-3]
    cands = cands[torch.linspace(0, len(cands) - 1, min(len(cands), 600)).long()]
    best, best_key = None, None
    B = margin.shape[0]
    for d in cands.tolist():
        hit = margin < d
        done = hit.any(1)
        n = int(done.sum())
        if not 0 < n < B:
            continue
        key = (len(set(hit.float().argmax(1)[done].tolist())), -abs(n / B - 0.6))
        if best_key is None or key > best_key:
            best, best_key = d, key
    if best is None:
        pytest.fail("no delta leaves some images finished and some not")
    return best


def _seq_sum(lp):
    """The f32 sum of per-token log-probs in step order, for every beam at once: (..., T) -> (...)."""
    s = torch.zeros(lp.shape[:-1], dtype=torch.float32, device=lp.device)
    for t in range(lp.shape[-1]):
        s = s + lp[..., t]
    return s


def _finish(tokens):
    """Step of each beam's first EOS (token column f + 1), -1 if none: (..., 1+T) -> (...)."""
    hit = tokens[..., 1:] == EOS
    return torch.where(hit.any(-1), hit.int().argmax(-1), torch.full(hit.shape[:-1], -1, device=tokens.device))


def _forced_logits(eng, memory_rows, tokens, T, **kw):
    """One teacher-forced decode call over [0, T) of `tokens` (N, 1+T): logits (N, T, V)."""
    ckv = eng.cross_kv(memory_rows)
    logits = torch.empty((tokens.shape[0], T, eng.dims.vocab), dtype=torch.float32, device=DEV)
    eng.decode(ckv, tokens.contiguous(), 0, T, max_tokens=T, forced=True, logits=logits, logits_row_offset=0, **kw)
    return logits


# ---- the premise ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision,opts", [("bf16", {}), ("bf16", {"per_op_kernels": True}), ("fp32", {"per_op_kernels": True})])
def test_one_step_forced_windows_equal_one_forced_call(model_p, precision, opts):
    model_p.set_precision(precision)
    B, T = 37, 40
    x = cases.images(B, seed=17).to(DEV)
    with M.decode_options(**opts):
        tokens, _ = model_p.generate_tokens(x, T, use_graph=False)
        eng = model_p._engine()
        _, memory = eng.encode(x, want_enc_out=False, want_memory=True)
        want = _forced_logits(eng, memory, tokens, T)
        ckv = eng.cross_kv(memory)
        got = torch.empty_like(want)
        kv, scratch = None, None
        for t in range(T):
            kv, scratch = eng.decode(ckv, tokens, t, t + 1, max_tokens=T, forced=True, logits=got, logits_row_offset=0, kv=kv,
                                     scratch=scratch)
    assert torch.equal(got, want)


# ---- fp32: tokens equal the oracle's ------------------------------------------------------------------------------------------
# seeds tried in order; the first whose oracle run keeps every selection margin above MARGIN is compared.  Over 98 steps the K-th and
# (K+1)-th candidates of these random-init models come within 1e-3 of each other for nearly every seed; 1e-4 is still 10x the fp32
# logit error.
SEEDS = [1000, 1001, 1002, 1003, 1004, 1005, 1006, 1007]
MARGIN = 1e-4
FP32_CASES = [(c, K, T) for c in ("P", "S") for K in (1, 3, 4) for T in (24, 98)] + [("T", 4, 24)]


@pytest.mark.parametrize("config,K,T", FP32_CASES)
def test_fp32_beam_equals_oracle(request, config, K, T):
    model = request.getfixturevalue({"P": "model_p", "S": "model_s", "T": "model_t"}[config])
    sd, cfg = cases.state_dict_of(model.cpu()), cases.oracle_cfg(config)
    model.to(DEV).set_precision("fp32")
    for seed in SEEDS:
        x = cases.images(2, seed=seed)
        want_t, want_s, want_l, margin = generate_beam(sd, x, cfg, T, K)
        if margin > MARGIN:
            break
    else:
        pytest.fail(f"no seed of {SEEDS} keeps the oracle's selection margins above {MARGIN}")
    tok, norm, lp, conf = model.generate_beam_tokens(x.to(DEV), T, K, eos_token=EOS)
    assert torch.equal(tok.cpu().long(), want_t), (seed, margin)
    assert (norm.cpu() - want_s).abs().max().item() <= 1e-4
    assert (lp.cpu() - want_l).abs().max().item() <= 1e-4


# ---- bf16 ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("opts", [{}, {"per_op_kernels": True}])
def test_bf16_one_beam_is_greedy(model_p, opts):
    model_p.set_precision("bf16")
    B, T = 16, 98
    x = cases.images(B, seed=23).to(DEV)
    with M.decode_options(**opts):
        want, want_c, lg = model_p.generate_tokens(x, T, return_logits=True, use_graph=False)
        top2 = lg.topk(2, dim=-1).values
        assert (top2[..., 0] - top2[..., 1]).min().item() > 1e-4       # no near-tie that log-softmax rounding could turn into a tie
        tok, norm, lp, conf = model_p.generate_beam_tokens(x, T, 1, eos_token=EOS)
    assert torch.equal(tok[:, 0], want)
    assert (conf[:, 0] - want_c).abs().max().item() <= 1e-5


def test_bf16_logprobs_match_the_oracle(model_p):
    """K = 4, T = 98, B = 16: each returned beam's per-token log-probs against the oracle's teacher-forced log-probs of that same
    sequence (2x the 2e-2 logit contract); scores are the sequential f32 sums of the returned log-probs, bit for bit."""
    sd, cfg = cases.state_dict_of(model_p.cpu()), cases.oracle_cfg("P")
    model_p.to(DEV).set_precision("bf16")
    B, K, T = 16, 4, 98
    x = cases.images(B, seed=29)
    tok, norm, lp, conf = model_p.generate_beam_tokens(x.to(DEV), T, K, eos_token=EOS)
    tok, norm, lp = tok.cpu().long(), norm.cpu(), lp.cpu()
    seqs = tok.view(B * K, T + 1)[:, :T]
    with torch.no_grad():
        enc = O.encoder_forward(sd, x, cfg).repeat_interleave(K, 0)
        h = sd["decoder.embedding.weight"][seqs] + sd["decoder.decoder_pos_embed"][:, :T]
        y = O.decoder_stack(sd, h, enc + sd["decoder.encoder_pos_embed"], seqs, cfg)
        lg = y @ sd["decoder.output.weight"].T + sd["decoder.output.bias"]
        want = torch.log_softmax(lg.float(), -1).gather(-1, tok.view(B * K, T + 1)[:, 1:, None])[..., 0].view(B, K, T)
    f = _finish(tok)
    live = torch.arange(T)[None, None, :] <= torch.where(f >= 0, f, torch.full_like(f, T))[..., None]
    err = (lp - want).abs()[live].max().item()
    print(f"bf16 K=4 T=98 B=16: per-token log-prob max|d| vs the oracle = {err:.3e}")
    assert err <= 4e-2
    lens = torch.where(f >= 0, f + 1, torch.full_like(f, T)).float()
    assert torch.equal(norm, _seq_sum(lp) / lens)


def test_kv_reorder_matches_a_fresh_forced_pass(model_p):
    """T = 40 crosses pages 0, 1 and 2, each shared and copied: the returned beams' per-token log-probs equal those of one teacher-
    forced decode call over the same tokens, which involves no reorder."""
    model_p.set_precision("bf16")
    B, K, T = 6, 4, 40
    x = cases.images(B, seed=31).to(DEV)
    tok, norm, lp, conf = model_p.generate_beam_tokens(x, T, K, eos_token=EOS)
    eng = model_p._engine()
    _, memory = eng.encode(x, want_enc_out=False, want_memory=True)
    lg = _forced_logits(eng, memory.repeat_interleave(K, 0), tok.view(B * K, T + 1), T)
    want = torch.log_softmax(lg, -1).gather(-1, tok.view(B * K, T + 1)[:, 1:, None].long())[..., 0].view(B, K, T)
    f = _finish(tok)
    live = torch.arange(T, device=DEV)[None, None, :] <= torch.where(f >= 0, f, torch.full_like(f, T))[..., None]
    assert (lp - want).abs()[live].max().item() <= 1e-5


# the per-operation chain switches its linears to the streaming form at 16 rows (decode.cu stream_linears), a different summation
# order: there the small batch is 4 images = 16 beam rows, on the same side of that switch as the batch of 37
@pytest.mark.parametrize("opts,lo,hi", [({}, 5, 6), ({"per_op_kernels": True}, 4, 8)])
def test_beam_is_batch_invariant_and_replays_equal(model_p, opts, lo, hi):
    model_p.set_precision("bf16")
    T, K = 24, 4
    x = cases.images(37, seed=37).to(DEV)
    with M.decode_options(**opts):
        part = model_p.generate_beam_tokens(x[lo:hi].contiguous(), T, K, eos_token=EOS)
        all_ = model_p.generate_beam_tokens(x, T, K, eos_token=EOS)
        again = model_p.generate_beam_tokens(x, T, K, eos_token=EOS)
    for a, b, c in zip(part, all_, again):
        assert torch.equal(a, b[lo:hi]) and torch.equal(b, c)


def test_eos_freezes_beams_and_length_penalty_orders(model_p):
    model_p.set_precision("bf16")
    B, K, T = 12, 4, 40
    x = cases.images(B, seed=43).to(DEV)
    delta = choose_delta(model_p, x, T)
    tokz = M.Tokenizer()
    with eos_bias(model_p, delta):
        for alpha in (1.0, 0.5):
            tok, norm, lp, conf = model_p.generate_beam_tokens(x, T, K, alpha, eos_token=EOS)
            f = _finish(tok)
            done = f[f >= 0].tolist()
            assert 0 < len(done) < B * K and len(set(done)) > 2, f
            for b in range(B):
                for k in range(K):
                    e = int(f[b, k])
                    if e < 0:
                        continue
                    assert (tok[b, k, e + 2:] == PAD).all() and (lp[b, k, e + 1:] == 0).all()
                    first_zero = e // 4 + 1
                    assert (conf[b, k, first_zero:] == 0).all()
            lens = torch.where(f >= 0, f + 1, torch.full_like(f, T)).float()
            raw = _seq_sum(lp)                                                  # the score never moves after EOS
            want = raw / lens ** torch.tensor(alpha, device=DEV)
            assert torch.allclose(norm, want, rtol=1e-6, atol=0)
            assert (norm[:, :-1] >= norm[:, 1:]).all()
            if alpha == 1.0:
                assert torch.equal(norm, raw / lens)
        out = M.generate_beam(model_p, x, tokz, max_len=T, num_beams=K)
    assert out[0].shape == (B, T + 1) and len(out[1]) == (T + 3) // 4
    bboxes, labels, confs = M.postprocess(*out, tokz)
    assert len(bboxes) == len(labels) == len(confs) == B


def test_beam_rejections(model_p):
    model_p.set_precision("bf16")
    x = cases.images(2, seed=5).to(DEV)
    tokz = M.Tokenizer()
    for K in (0, 17):
        with pytest.raises(ValueError):
            model_p.generate_beam_tokens(x, 8, K, eos_token=EOS)
        with pytest.raises(ValueError):
            M.generate_beam(model_p, x, tokz, max_len=8, num_beams=K)
    with pytest.raises(ValueError):
        model_p.generate_beam_tokens(x, 8, 2, eos_token=305)
    with pytest.raises(RuntimeError):
        model_p.generate_beam_tokens(x, 100, 2, eos_token=EOS)
    with pytest.raises(ValueError):
        M.generate_beam(model_p, x, tokz, max_len=100)
    with pytest.raises(ValueError):
        M.generate_beam(model_p, x.cpu(), tokz, max_len=8)
    # the C ABI itself
    from mdcnet_b200.model import BeamPlan
    eng = model_p._engine()
    plan = BeamPlan(eng, 2, 8, 2, 1.0, EOS, use_graph=False)
    plan.run(x)                                             # a valid state and logits to step from
    lib, s = eng.lib, L.stream_ptr(DEV)
    assert lib.mdc_beam_workspace_bytes(eng.handle, 2, 17) == 0 and lib.mdc_beam_workspace_bytes(eng.handle, 2, 0) == 0

    def step(**kw):
        st = L.BeamState.from_buffer_copy(plan.state)
        for k, v in kw.items():
            setattr(st, k, v)
        return lib.mdc_beam_step(eng.handle, C.byref(st), C.c_void_p(plan.logits.data_ptr()), 8 * eng.dims.vocab, 0, s)

    assert step() == 0
    for bad in ({"K": 0}, {"K": 17}, {"eos_token": 305}, {"eos_token": -1}, {"workspace_bytes": plan.state.workspace_bytes - 1}):
        assert step(**bad) != 0, bad
        assert lib.mdc_last_error().decode()
    st = L.BeamState.from_buffer_copy(plan.state)
    assert lib.mdc_beam_step(eng.handle, C.byref(st), C.c_void_p(plan.logits.data_ptr()), 8 * eng.dims.vocab, eng.dims.max_pos, s) != 0
    assert lib.mdc_beam_step(eng.handle, C.byref(st), C.c_void_p(plan.logits.data_ptr()), 8 * eng.dims.vocab, 8, s) != 0   # token columns
    torch.cuda.synchronize()
