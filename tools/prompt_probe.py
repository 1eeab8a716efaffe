"""Cost of prompted generation (generate_tokens(..., prompt=)) on configs P and T, B = 64, bf16, T = 99 new columns.

Per config, graph-replayed calls, alternated `--reps` times: the unprompted call; a 16-token prompt on every row run as 16 decode steps
(decode_options(prefill=False)) and as one all-positions prefill pass followed by the remaining steps; and, for the prefill threshold,
prompts of n = 1, 2, 3, 4, 6, 8 and 16 tokens both ways.  The threshold is the smallest n from which the prefill is faster at every
measured n on both configs.

  python tools/prompt_probe.py --out RESULT.json [--configs P,T] [--reps 3] [--iters 20]
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
from mdcnet_b200 import model as MM  # noqa: E402
from oracle import cases  # noqa: E402

B, T = 64, 99
NS = [1, 2, 3, 4, 6, 8, 16]


def prompt_of(n, seed):
    g = torch.Generator().manual_seed(seed)
    p = torch.randint(270, 299, (B, n), generator=g)
    p[:, 0], p[:, -1] = 303, 304
    return p


def ms_per_call(fn, iters):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / iters * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="P,T")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", required=True, help="JSON file for the results (GPU name and power limit included)")
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip(), "B": B, "T": T, "reps": a.reps, "iters": a.iters,
           "unit": "ms per generate_tokens call (graph replay, encoder included)", "configs": {}}
    print(res["gpu"], "|", res["nvidia_smi"], flush=True)
    MM.PREFILL_MIN_STEPS = 1          # measure the prefill at every n; the shipped threshold is what this probe justifies
    for config in a.configs.split(","):
        m = cases.build_product_model(config, seed=0, gamma_seed=5).to("cuda").set_precision("bf16")
        x = cases.images(B, seed=1000).to("cuda")
        prompts = {n: prompt_of(n, n) for n in NS}
        runs = {"unprompted": lambda: m.generate_tokens(x, T)}
        for n in NS:
            for prefill in (False, True):
                def run(n=n, prefill=prefill):
                    with M.decode_options(prefill=prefill):
                        m.generate_tokens(x, T, prompt=prompts[n])
                runs[f"n{n}_{'prefill' if prefill else 'steps'}"] = run
        times = {k: [] for k in runs}
        for _ in range(a.reps):
            for k, fn in runs.items():
                times[k].append(ms_per_call(fn, a.iters))
        best = {k: min(v) for k, v in times.items()}
        # the prefilled prompt gives the same tokens as the step path up to rounding: report how many of the 64 x 99 columns agree
        with M.decode_options(prefill=False):
            ts, _ = m.generate_tokens(x, T, prompt=prompts[16])
        with M.decode_options(prefill=True):
            tp, _ = m.generate_tokens(x, T, prompt=prompts[16])
        res["configs"][config] = {"ms_all_reps": times, "ms_best": best,
                                  "n16_token_agreement": float((ts == tp).float().mean())}
        print(config, json.dumps({k: round(v, 3) for k, v in best.items()}), flush=True)
        del m
        torch.cuda.empty_cache()
    faster = {n: all(res["configs"][c]["ms_best"][f"n{n}_prefill"] < res["configs"][c]["ms_best"][f"n{n}_steps"] for c in res["configs"])
              for n in NS}
    res["prefill_faster_at"] = {str(n): v for n, v in faster.items()}
    res["threshold"] = next((n for i, n in enumerate(NS) if all(faster[k] for k in NS[i:])), None)
    print("threshold", res["threshold"], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
