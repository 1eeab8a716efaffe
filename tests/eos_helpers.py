"""Test helpers that make EOS arrive at varied, predictable steps without any test hook: adding a constant delta to the EOS bias makes
an image emit EOS at the first step whose margin max_{v != eos} logit_v - logit_eos (in the no-stop run of the unmodified model) is
below delta; the trajectory before that step is unchanged."""
import contextlib

import pytest
import torch

EOS = 301


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
