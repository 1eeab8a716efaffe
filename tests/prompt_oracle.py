"""Prompted generation on the CPU oracle: O.generate, except that row b's first l_b new tokens are its prompt (step t with t + 1 <= l_b
keeps prompt[b, t]; its confidence is the max probability of the filtered distribution at that step, as at any step).  The reference the
GPU prompt tests compare against."""
import torch

from oracle import mdc_oracle as O


def generate_prompted(sd, image, cfg, max_len, prompt, lengths, top_k=0, top_p=1.0, uniforms=None, return_logits=False):
    B = image.shape[0]
    prompt = torch.as_tensor(prompt).long().view(B, -1)
    lengths = torch.as_tensor(lengths).long().view(B)
    enc = O.encoder_forward(sd, image, cfg)
    toks = torch.full((B, 1), cfg.bos_idx, dtype=torch.long)
    confs, all_logits = [], []
    for i in range(max_len):
        logits = O.next_token_logits(sd, enc, toks, cfg)
        if return_logits:
            all_logits.append(logits)
        logits = O.top_k_top_p_filtering(logits, top_k=top_k, top_p=top_p)
        if i % 4 == 0:
            confs.append(torch.softmax(logits, dim=-1).max(dim=-1)[0])
        if top_k != 0 or top_p != 1:
            nxt = O.sample_from_uniform(logits, uniforms[:, i])
        else:
            nxt = torch.softmax(logits, dim=-1).argmax(dim=-1)
        if i < prompt.shape[1]:
            nxt = torch.where(i + 1 <= lengths, prompt[:, i], nxt)
        toks = torch.cat([toks, nxt.view(-1, 1)], dim=1)
    if return_logits:
        return toks, confs, torch.stack(all_logits, dim=1)
    return toks, confs
