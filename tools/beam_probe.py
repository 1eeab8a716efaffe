"""Throughput of beam search (EncoderDecoder.generate_beam_tokens), bf16, T = 99, on the seeded test models.

Rows: config P at B in {16, 64} x K in {1, 2, 4, 8}, and the trained geometry T at B = 16 x K in {1, 4}.  Beside each row, greedy
generate_tokens at B images and at B*K images (the same number of decoded rows).  img/s counts images (not beams), over `--reps`
graph replays after two warm-up calls, the three measurements alternating.  The card's name and power limit are read in the same run,
and each row records the library launches of one beam call.  Reported, not a pass/fail gate.

  python tools/beam_probe.py --out RESULT.json [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mdcnet_b200 as M  # noqa: E402
from oracle import cases  # noqa: E402

EOS, T = 301, 99
ROWS = [("P", B, K) for B in (16, 64) for K in (1, 2, 4, 8)] + [("T", 16, K) for K in (1, 4)]


def timed_ips(fn, B, reps):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return B * reps / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    card = q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"
    models = {c: cases.build_product_model(c, seed=0, gamma_seed=5).to("cuda").set_precision("bf16") for c in ("P", "T")}
    rows = []
    for config, B, K in ROWS:
        model = models[config]
        x = cases.images(B * K, seed=7).to("cuda")
        xb = x[:B].contiguous()
        beam = lambda: model.generate_beam_tokens(xb, T, K, eos_token=EOS)
        greedy_b = lambda: model.generate_tokens(xb, T)
        greedy_bk = lambda: model.generate_tokens(x, T)
        beam()
        n0 = M._lib.launch_count()
        beam()
        launches = M._lib.launch_count() - n0
        res = {"beam": [], "greedy_B": [], "greedy_BK": []}
        for _ in range(2):
            res["beam"].append(timed_ips(beam, B, args.reps))
            res["greedy_B"].append(timed_ips(greedy_b, B, args.reps))
            res["greedy_BK"].append(timed_ips(greedy_bk, B * K, args.reps))
        row = {"config": config, "B": B, "K": K, "T": T, "launches_per_beam_call": launches,
               **{k + "_img_s": round(max(v), 1) for k, v in res.items()}}
        row["beam_over_greedy_B"] = round(row["beam_img_s"] / row["greedy_B_img_s"], 3)
        print(json.dumps(row), flush=True)
        rows.append(row)
        for plans in (model.__dict__.get("_plans", {}),):
            for k in [k for k in plans if k != "eng"]:
                del plans[k]                  # free the graphs and buffers of this shape before the next
        torch.cuda.empty_cache()
    out = {"card": card, "precision": "bf16", "T": T, "reps": args.reps, "rows": rows,
           "note": "img/s = images per second (all K beams of an image count once); greedy_BK decodes B*K images"}
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("card:", card)


if __name__ == "__main__":
    main()
