"""CPU: the reference prompted beam search (tests/prompt_beam_oracle.py) and the host checks of prompted beam search.

Without prompt tokens it is tests/beam_oracle.generate_beam exactly; with one beam its tokens are the prompted greedy oracle's.  The
prompt columns are kept with log-prob 0, a score stays the sequential f32 sum of the per-token log-probs, and the length normalisation
counts generated tokens only.  check_beam_prompt rejects what the kernels must never see, including a prompt that leaves no step."""
import pytest
import torch

from mdcnet_b200.model import check_beam_prompt
from oracle import cases
from tests import beam_oracle
from tests.prompt_beam_oracle import generate_beam
from tests.prompt_oracle import generate_prompted

EOS, PAD, SOC, EOC = 301, 302, 303, 304


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


def _prompts(B, P, lengths, seed):
    g = torch.Generator().manual_seed(seed)
    prompt = torch.randint(270, 299, (B, P), generator=g)
    prompt[:, 0] = SOC
    for b, l in enumerate(lengths):
        prompt[b, l:] = PAD
    return prompt


@pytest.mark.parametrize("config,K", [("S", 3), ("P", 4)])
def test_zero_lengths_are_the_unprompted_search(config, K):
    sd, cfg = _setup(config, 1.5)
    x = cases.images(2, seed=43)
    T = 8
    want = beam_oracle.generate_beam(sd, x, cfg, T, K)
    got = generate_beam(sd, x, cfg, T, K, prompt=torch.full((2, 3), 280), lengths=[0, 0])
    for a, b in zip(got[:3], want[:3]):
        assert torch.equal(a, b)
    assert got[3] == want[3]


@pytest.mark.parametrize("config", ["S", "P"])
def test_one_beam_is_prompted_greedy(config):
    sd, cfg = _setup(config)
    x = cases.images(3, seed=44)
    T, lengths = 9, [0, 3, 6]
    prompt = _prompts(3, 6, lengths, 1)
    want, _ = generate_prompted(sd, x, cfg, T, prompt, lengths)
    tok, _, _, margin = generate_beam(sd, x, cfg, T, 1, prompt=prompt, lengths=lengths)
    assert margin > 0
    assert torch.equal(tok[:, 0], want)


def test_prompt_columns_logprobs_and_scores():
    sd, cfg = _setup("S", 1.5)
    B, K, T = 3, 3, 9
    lengths = [2, 0, 5]
    x = cases.images(B, seed=45)
    prompt = _prompts(B, 5, lengths, 2)
    _, want_c = generate_prompted(sd, x, cfg, T, prompt, lengths)
    tok, score, lp, margin, conf = generate_beam(sd, x, cfg, T, K, 0.0, prompt=prompt, lengths=lengths, return_confs=True)
    assert margin > 0
    n_fin = 0
    for b, l in enumerate(lengths):
        assert (tok[b, :, 1:1 + l] == prompt[b, :l]).all()           # every beam carries the prompt
        assert (lp[b, :, :l] == 0).all()                             # prompt steps score nothing
        for t in range(0, l, 4):                                     # prompt-step confidences: the prompted greedy step's
            assert torch.allclose(conf[b, :, t // 4], want_c[t // 4][b].expand(K), rtol=1e-6, atol=0)
        for k in range(K):
            assert torch.equal(score[b, k], _seq_sum(lp[b, k]))       # length_penalty 0: the raw score
            assert (lp[b, k, l:] <= 0).all()
            n_fin += bool((tok[b, k, 1:] == EOS).any())
    assert 0 < n_fin < B * K, "the EOS bias should finish some beams and not others"


@pytest.mark.parametrize("alpha", [1.0, 0.5])
def test_normalised_score_counts_generated_tokens(alpha):
    sd, cfg = _setup("S", 2.0)
    B, K, T = 2, 3, 8
    lengths = [4, 1]
    x = cases.images(B, seed=46)
    prompt = _prompts(B, 4, lengths, 3)
    tok, norm, lp, _ = generate_beam(sd, x, cfg, T, K, alpha, prompt=prompt, lengths=lengths)
    for b, l in enumerate(lengths):
        for k in range(K):
            hits = (tok[b, k, 1:] == EOS).nonzero()
            n = int(hits[0]) + 1 - l if len(hits) else T - l
            assert n >= 1
            want = _seq_sum(lp[b, k]) / torch.tensor(float(n)) ** torch.tensor(alpha)
            assert torch.allclose(norm[b, k], want, rtol=1e-6, atol=0)
            if alpha == 1.0:
                assert torch.equal(norm[b, k], want)
        assert all(norm[b, j] >= norm[b, j + 1] for j in range(K - 1))


def test_check_beam_prompt():
    vocab, T = 305, 6
    p = torch.tensor([[SOC, 280, EOC, 7], [SOC, 281, 282, EOC]])
    out, lens = check_beam_prompt(p, [3, 4], 2, T, vocab, EOS)
    assert out.dtype == torch.int32 and out.tolist() == [[SOC, 280, EOC, PAD], [SOC, 281, 282, EOC]] and lens.tolist() == [3, 4]
    out, lens = check_beam_prompt(p, [3, 4], 2, 5, vocab, EOS)         # l_b = T - 1: one free step
    assert lens.tolist() == [3, 4]
    bad = [
        (torch.tensor([[SOC, PAD]]), [2], 1, T),                   # PAD inside the prompt
        (torch.tensor([[SOC, EOS]]), [2], 1, T),                   # EOS inside the prompt
        (torch.tensor([[SOC, vocab]]), [2], 1, T),                 # outside the vocabulary
        (torch.tensor([[SOC, -1]]), [2], 1, T),
        (torch.tensor([[SOC, 280]]), [3], 1, T),                   # l_b > P
        (torch.tensor([[SOC, 280]]), [-1], 1, T),
        (torch.tensor([[SOC, 280]]), [2], 1, 2),                   # l_b = T: no step left to search
        (torch.tensor([[SOC, 280]]), [2], 1, 1),                   # l_b > T
        (torch.tensor([[SOC, 280]]), [2, 2], 2, T),                # batch mismatch
        (torch.tensor([SOC, 280]), [2], 1, T),                     # not (B, P)
        (torch.tensor([[0.5, 1.0]]), [2], 1, T),                   # not integers
        (None, [2], 1, T),                                         # lengths without a prompt
    ]
    for prompt, lengths, B, TT in bad:
        with pytest.raises(ValueError):
            check_beam_prompt(prompt, lengths, B, TT, vocab, EOS)
    check_beam_prompt(torch.tensor([[SOC, 280]]), None, 1, 3, vocab, EOS)      # default l_b = P = T - 1
    with pytest.raises(ValueError):
        check_beam_prompt(torch.tensor([[SOC, 280]]), None, 1, 2, vocab, EOS)  # default l_b = P = T
    with pytest.raises(ValueError):
        check_beam_prompt(torch.tensor([[SOC, 7]]), [2], 1, T, vocab, 7)       # the caller's EOS, not only 301
