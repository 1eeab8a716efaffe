"""CPU: the reference beam search (tests/beam_oracle.py, on the oracle's decoder), the reference the GPU beam tests compare against.

It must reduce to greedy generate() at one beam, keep each beam's score equal to the f32 sum of its per-token log-probs in step order,
freeze finished beams (PAD after EOS, log-prob 0, score unchanged) and return beams ordered by normalised score.  EOS is made to arrive
within a few steps by raising its output bias."""
import pytest
import torch

from oracle import cases, mdc_oracle as O
from tests.beam_oracle import generate_beam

EOS, PAD = 301, 302


def _setup(config, eos_delta=0.0):
    model = cases.build_product_model(config, seed=0, gamma_seed=5)
    sd, cfg = cases.state_dict_of(model), cases.oracle_cfg(config)
    sd["decoder.output.bias"][EOS] += eos_delta
    return sd, cfg


def _seq_sum(lp):
    s = torch.zeros((), dtype=torch.float32)
    for v in lp:
        s = s + v
    return s


def _lengths(tokens, T):
    """f + 1 for a beam whose first EOS is at step f (token column f + 1), else T."""
    out = []
    for row in tokens.tolist():
        hits = [i for i, v in enumerate(row[1:]) if v == EOS]
        out.append(hits[0] + 1 if hits else T)
    return out


@pytest.mark.parametrize("config", ["S", "P"])
def test_one_beam_is_greedy(config):
    sd, cfg = _setup(config)
    x = cases.images(2, seed=41)
    T = 6
    want, _ = O.generate(sd, x, cfg, max_len=T)
    tok, score, lp, _ = generate_beam(sd, x, cfg, T, 1)
    assert torch.equal(tok[:, 0], want)


@pytest.mark.parametrize("config,K,delta", [("S", 3, 2.0), ("P", 4, 1.5)])
def test_beam_scores_rescore_and_freeze(config, K, delta):
    sd, cfg = _setup(config, delta)
    x = cases.images(2, seed=43)
    T, alpha = 8, 1.0
    tok, norm, lp, margin = generate_beam(sd, x, cfg, T, K, alpha)
    assert tok.shape == (2, K, T + 1) and norm.shape == (2, K) and lp.shape == (2, K, T)
    assert margin > 0
    n_fin = 0
    enc = O.encoder_forward({k: v.float() for k, v in sd.items()}, x, cfg)
    for b in range(2):
        lens = _lengths(tok[b], T)
        for k in range(K):
            # score = the sequential f32 sum of the per-token log-probs, normalised by len^alpha
            assert torch.equal(norm[b, k], _seq_sum(lp[b, k]) / torch.tensor(float(lens[k])) ** torch.tensor(alpha))
            if lens[k] < T:                                   # finished: PAD after EOS, log-prob 0 after it
                n_fin += 1
                f = lens[k] - 1
                assert (tok[b, k, f + 2:] == PAD).all() and (lp[b, k, f + 1:] == 0).all()
            # a fresh teacher-forced rescoring of the returned sequence gives the same per-token log-probs
            for t in range(lens[k]):
                lg = O.next_token_logits(sd, enc[b:b + 1], tok[b, k:k + 1, :t + 1], cfg).float()[0]
                want = torch.log_softmax(lg, -1)[tok[b, k, t + 1]]
                assert abs(float(want) - float(lp[b, k, t])) <= 1e-5, (b, k, t)
        assert all(norm[b, j] >= norm[b, j + 1] for j in range(K - 1))       # best first
    assert 0 < n_fin < 2 * K, "the EOS bias should finish some beams and not others"


def test_length_penalty_orders_by_formula():
    sd, cfg = _setup("S", 2.0)
    x = cases.images(2, seed=43)
    T = 8
    for alpha in (0.0, 2.0):
        tok, norm, lp, _ = generate_beam(sd, x, cfg, T, 3, alpha)
        for b in range(2):
            lens = _lengths(tok[b], T)
            raw = [float(_seq_sum(lp[b, k])) for k in range(3)]
            want = [r / l ** alpha for r, l in zip(raw, lens)]
            assert want == sorted(want, reverse=True)
            assert torch.allclose(norm[b], torch.tensor(want), rtol=1e-6, atol=0)
