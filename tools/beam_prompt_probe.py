"""Cost of prompted beam search (generate_beam_tokens(..., prompt=)), bf16, K = 4 beams, T = 99 columns, 16-token caption prompts.

Configs: P at B = 64 and T at B = 16.  Per config, graph-replayed calls with the encoder included, the three cases alternated `--reps`
times, best of the repetitions: the unprompted search; the prompt run as 16 decode windows with their beam steps
(decode_options(prefill=False)); the prompt prefilled over the B*K rows in one all-positions pass, then the windows from step 16.  Beside
them the prefill pass's own time: the pass alone (mdc_decode_prefill_steps over the B*K rows, confidences on), captured as a CUDA graph
and timed with CUDA events.  The card's name and power limit are read in the same run.

  python tools/beam_prompt_probe.py --out RESULT.json [--configs P,T] [--reps 3] [--iters 10]
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

EOS, K, T, N = 301, 4, 99, 16
BATCH = {"P": 64, "T": 16}


def caption_prompts(B, seed):
    g = torch.Generator().manual_seed(seed)
    p = torch.randint(270, 299, (B, N), generator=g)
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


def prefill_pass_ms(m, B, iters):
    """The prefill pass of the cached prefilled plan, alone: its own buffers, one CUDA graph, CUDA events around `iters` replays."""
    plan = next(p for k, p in m.__dict__["_plans"].items() if k != "eng" and isinstance(p, MM.BeamPlan) and p.prefill == N and p.B == B)
    eng = plan.eng

    def launch():
        eng.decode(plan.ckv, plan.tokens, 0, N, max_tokens=T, forced=False, confs=plan.confs, kv=plan.kv, scratch=plan.scratch,
                   prefill=N, prefill_ws=plan.prefill_ws)

    [captured] = MM.capture_graphs(eng.device, launch)
    best = float("inf")
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        MM.replay(eng.device, captured)
        e0.record()
        for _ in range(iters):
            MM.replay(eng.device, captured)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / iters)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="P,T")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", required=True, help="JSON file for the results (GPU name and power limit included)")
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip(), "precision": "bf16", "K": K, "T": T, "prompt_tokens": N,
           "reps": a.reps, "iters": a.iters, "unit": "ms per generate_beam_tokens call (graph replay, encoder included)", "configs": {}}
    print(res["gpu"], "|", res["nvidia_smi"], flush=True)
    for config in a.configs.split(","):
        B = BATCH[config]
        m = cases.build_product_model(config, seed=0, gamma_seed=5).to("cuda").set_precision("bf16")
        x = cases.images(B, seed=1000).to("cuda")
        prompt = caption_prompts(B, 16)

        def run(prompted, prefill):
            with M.decode_options(prefill=prefill):
                if prompted:
                    return m.generate_beam_tokens(x, T, K, eos_token=EOS, prompt=prompt)
                return m.generate_beam_tokens(x, T, K, eos_token=EOS)

        runs = {"unprompted": lambda: run(False, True), "prompt_steps": lambda: run(True, False), "prompt_prefill": lambda: run(True, True)}
        times = {k: [] for k in runs}
        for _ in range(a.reps):
            for k, fn in runs.items():
                times[k].append(ms_per_call(fn, a.iters))
        best = {k: min(v) for k, v in times.items()}
        n0 = M._lib.launch_count()
        runs["prompt_prefill"]()
        launches_prefill = M._lib.launch_count() - n0
        n0 = M._lib.launch_count()
        runs["prompt_steps"]()
        launches_steps = M._lib.launch_count() - n0
        pass_ms = prefill_pass_ms(m, B, 50)
        # the prefilled prompt against the step path: how many returned beams are the same token sequence
        ts, tp = runs["prompt_steps"]()[0], runs["prompt_prefill"]()[0]
        same = (ts == tp).all(-1).float().mean().item()
        res["configs"][config] = {"B": B, "ms_all_reps": times, "ms_best": best, "prefill_pass_ms": pass_ms,
                                  "prefill_pass_share_of_prefilled_call": pass_ms / best["prompt_prefill"],
                                  "launches_per_call": {"prompt_steps": launches_steps, "prompt_prefill": launches_prefill},
                                  "beams_equal_prefill_vs_steps": same}
        print(config, json.dumps({**{k: round(v, 3) for k, v in best.items()}, "prefill_pass_ms": round(pass_ms, 3),
                                  "beams_equal": same}), flush=True)
        del m
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
