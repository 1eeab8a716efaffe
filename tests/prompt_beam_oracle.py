"""Reference prompted beam search for the prompted beam tests: tests/beam_oracle.generate_beam, except that every beam of image b starts
from BOS followed by prompt[b, :l_b] (include/mdc_b200.h "Prompted beam search", DESIGN.md §3.4c).  Step t with t + 1 <= l_b selects
nothing for image b: its K rows keep the prompt token in column t+1 and a log-prob of 0, beam 0 stays the only running beam.  Step l_b is
the first beam step.  Length normalisation counts generated tokens only.  Float32 on the oracle's prefix-only decoder.  Test
infrastructure only."""
import numpy as np
import torch

from oracle import mdc_oracle as O
from oracle.mdc_oracle import OracleCfg


def generate_beam(sd, image, cfg: OracleCfg, max_len, num_beams, length_penalty=1.0, eos=301, prompt=None, lengths=None,
                  return_confs=False):
    """Returns tokens long (B, K, 1+T), normalised scores f32 (B, K), per-token log-probs f32 (B, K, T), each image's beams best first,
    and the smallest selection margin of any free step or final ordering (as tests/beam_oracle.generate_beam).  With `return_confs`
    also the confidences f32 (B, K, ceil(T/4)): at a prompt step the max probability of beam 0's distribution, at a free step exp(lp)
    of the chosen candidate (0 after a beam's EOS)."""
    B, K, T = image.shape[0], int(num_beams), int(max_len)
    if prompt is None:
        prompt, lengths = torch.zeros((B, 0), dtype=torch.long), torch.zeros(B, dtype=torch.long)
    prompt = torch.as_tensor(prompt).long().view(B, -1)
    lengths = torch.as_tensor(lengths).long().view(B)
    assert int(lengths.max()) <= T - 1, "beam search needs a free step after the prompt"
    sd = {k: v.float() for k, v in sd.items()}
    enc = O.encoder_forward(sd, image.float(), cfg).repeat_interleave(K, dim=0)
    toks = torch.full((B * K, 1 + T), cfg.pad_idx, dtype=torch.long)
    toks[:, 0] = cfg.bos_idx
    for b in range(B):
        toks[b * K:(b + 1) * K, 1:1 + int(lengths[b])] = prompt[b, :int(lengths[b])]
    score = torch.full((B, K), -float("inf"), dtype=torch.float32)
    score[:, 0] = 0.0
    fin = torch.full((B, K), -1, dtype=torch.long)
    lps = torch.zeros((B * K, T), dtype=torch.float32)
    confs = torch.zeros((B * K, (T + 3) // 4), dtype=torch.float32)
    margin = float("inf")
    for t in range(T):
        lg = O.next_token_logits(sd, enc, toks[:, :t + 1], cfg).float()
        m = lg.max(-1, keepdim=True).values
        lp = (lg - m) - torch.log(torch.exp(lg - m).sum(-1, keepdim=True))
        new_toks, new_lps, new_confs = toks.clone(), lps.clone(), confs.clone()
        new_score, new_fin = score.clone(), fin.clone()
        for b in range(B):
            if t + 1 <= int(lengths[b]):                      # a prompt step: nothing selected, nothing moved
                if t % 4 == 0:
                    new_confs[b * K, t // 4] = torch.softmax(lg[b * K], -1).max()
                continue
            c_score, c_k, c_v, c_lp = [], [], [], []
            for k in range(K):
                r = b * K + k
                if fin[b, k] >= 0:
                    c_score.append(score[b, k:k + 1]); c_k.append(torch.tensor([k])); c_v.append(torch.tensor([cfg.pad_idx]))
                    c_lp.append(torch.zeros(1))
                elif score[b, k] > -float("inf"):
                    V = lp.shape[1]
                    c_score.append(score[b, k] + lp[r]); c_k.append(torch.full((V,), k)); c_v.append(torch.arange(V)); c_lp.append(lp[r])
            cs, ck, cv, cl = (torch.cat(x) for x in (c_score, c_k, c_v, c_lp))
            order = np.lexsort((cv.numpy(), ck.numpy(), -cs.double().numpy()))
            if len(order) > K:
                margin = min(margin, float(cs[order[K - 1]].double() - cs[order[K]].double()))
            for j, i in enumerate(order[:K].tolist()):
                p, v = b * K + int(ck[i]), int(cv[i])
                fp = int(fin[b, int(ck[i])])
                new_toks[b * K + j] = toks[p]
                new_toks[b * K + j, t + 1] = v
                new_lps[b * K + j] = lps[p]
                new_lps[b * K + j, t] = cl[i]
                new_confs[b * K + j] = confs[p]
                if t % 4 == 0:
                    new_confs[b * K + j, t // 4] = 0.0 if fp >= 0 else torch.exp(cl[i])
                new_score[b, j] = cs[i]
                new_fin[b, j] = fp if fp >= 0 else (t if v == eos else -1)
        toks, lps, confs, score, fin = new_toks, new_lps, new_confs, new_score, new_fin
    lb = lengths[:, None]
    length = torch.where(fin >= 0, fin + 1 - lb, T - lb).to(torch.float32)
    norm = score / length ** torch.tensor(float(length_penalty), dtype=torch.float32)
    out_t = torch.empty((B, K, 1 + T), dtype=torch.long)
    out_s = torch.empty((B, K), dtype=torch.float32)
    out_l = torch.empty((B, K, T), dtype=torch.float32)
    out_c = torch.empty((B, K, confs.shape[1]), dtype=torch.float32)
    for b in range(B):
        order = sorted(range(K), key=lambda k: (-float(norm[b, k]), k))
        for j, k in enumerate(order):
            out_t[b, j], out_s[b, j], out_l[b, j], out_c[b, j] = toks[b * K + k], norm[b, k], lps[b * K + k], confs[b * K + k]
        for j in range(K - 1):
            margin = min(margin, float(out_s[b, j].double() - out_s[b, j + 1].double()))
    if return_confs:
        return out_t, out_s, out_l, margin, out_c
    return out_t, out_s, out_l, margin
