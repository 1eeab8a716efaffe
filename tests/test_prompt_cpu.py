"""CPU: the prompted oracle (tests/prompt_oracle.py) and the host side of prompted generation.

With no prompt tokens, or with a prompt equal to the row's own unprompted output, the prompted oracle is exactly O.generate; a foreign
prompt is kept verbatim.  Tokenizer.caption_prompt pads ragged captions, and check_prompt rejects what the kernels must never see."""
import pytest
import torch

import mdcnet_b200 as M
from mdcnet_b200.model import check_prompt
from oracle import cases, mdc_oracle as O
from tests.prompt_oracle import generate_prompted

PAD, EOS, SOC, EOC = 302, 301, 303, 304


def _setup(config):
    model = cases.build_product_model(config, seed=0, gamma_seed=5)
    return cases.state_dict_of(model), cases.oracle_cfg(config)


@pytest.mark.parametrize("top_k", [0, 5])
def test_no_prompt_is_generate(top_k):
    sd, cfg = _setup("S")
    B, T = 3, 9
    x = cases.images(B, seed=21)
    u = torch.rand(B, T, generator=torch.Generator().manual_seed(2))
    want_t, want_c = O.generate(sd, x, cfg, max_len=T, top_k=top_k, uniforms=u)
    prompt = torch.full((B, 4), 7, dtype=torch.long)          # ignored: every length is 0
    got_t, got_c = generate_prompted(sd, x, cfg, T, prompt, [0, 0, 0], top_k=top_k, uniforms=u)
    assert torch.equal(got_t, want_t)
    assert all(torch.equal(a, b) for a, b in zip(got_c, want_c))


@pytest.mark.parametrize("top_k", [0, 5])
def test_own_prefix_is_generate(top_k):
    sd, cfg = _setup("S")
    B, T = 3, 9
    x = cases.images(B, seed=22)
    u = torch.rand(B, T, generator=torch.Generator().manual_seed(3))
    want_t, want_c = O.generate(sd, x, cfg, max_len=T, top_k=top_k, uniforms=u)
    lengths = torch.tensor([0, 4, T])
    got_t, got_c = generate_prompted(sd, x, cfg, T, want_t[:, 1:], lengths, top_k=top_k, uniforms=u)
    assert torch.equal(got_t, want_t)
    assert all(torch.equal(a, b) for a, b in zip(got_c, want_c))


def test_foreign_prompt_is_kept():
    sd, cfg = _setup("S")
    B, T = 2, 8
    x = cases.images(B, seed=23)
    prompt = torch.tensor([[SOC, 280, 281, EOC], [SOC, 290, EOC, PAD]])
    toks, confs = generate_prompted(sd, x, cfg, T, prompt, [4, 3])
    assert toks[0, 1:5].tolist() == prompt[0].tolist() and toks[1, 1:4].tolist() == prompt[1, :3].tolist()
    assert len(confs) == (T + 3) // 4


def test_caption_prompt_padding():
    tok = M.Tokenizer()
    prompt, lengths = tok.caption_prompt([[280, 281, 282], [], [290]])
    assert prompt.tolist() == [[SOC, 280, 281, 282, EOC], [SOC, EOC, PAD, PAD, PAD], [SOC, 290, EOC, PAD, PAD]]
    assert lengths.tolist() == [5, 2, 3]
    with pytest.raises(ValueError):
        tok.caption_prompt([[280, EOS]])
    with pytest.raises(ValueError):
        tok.caption_prompt([])


def test_check_prompt():
    vocab = 305
    p = torch.tensor([[SOC, 280, EOC, 7], [SOC, 281, 282, EOC]])
    out, lens = check_prompt(p, [3, 4], 2, 10, vocab, EOS)
    assert out.dtype == torch.int32 and out.tolist() == [[SOC, 280, EOC, PAD], [SOC, 281, 282, EOC]] and lens.tolist() == [3, 4]
    out, lens = check_prompt(p, [3, 2], 2, 3, vocab, EOS)          # P > T: only the first T columns can be prompt columns
    assert out.tolist() == [[SOC, 280, EOC], [SOC, 281, PAD]] and lens.tolist() == [3, 2]
    bad = [
        (torch.tensor([[SOC, PAD]]), [2], 1, 10),                  # PAD inside the prompt
        (torch.tensor([[SOC, EOS]]), [2], 1, 10),                  # EOS inside the prompt
        (torch.tensor([[SOC, vocab]]), [2], 1, 10),                # outside the vocabulary
        (torch.tensor([[SOC, -1]]), [2], 1, 10),
        (torch.tensor([[SOC, 280]]), [3], 1, 10),                  # l_b > P
        (torch.tensor([[SOC, 280]]), [-1], 1, 10),
        (torch.tensor([[SOC, 280]]), [2], 1, 1),                   # l_b > T
        (torch.tensor([[SOC, 280]]), [2, 2], 2, 10),               # batch mismatch
        (torch.tensor([SOC, 280]), [2], 1, 10),
        (torch.tensor([[0.5, 1.0]]), [2], 1, 10),
    ]
    for prompt, lengths, B, T in bad:
        with pytest.raises(ValueError):
            check_prompt(prompt, lengths, B, T, vocab, EOS)
    check_prompt(torch.tensor([[SOC, PAD]]), [1], 1, 10, vocab, EOS)   # past the length: ignored
