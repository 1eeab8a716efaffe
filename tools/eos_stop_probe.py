"""Throughput of stop at EOS (generate(..., stop_at_eos=True)) on configs P and T, B = 64, bf16, T = 99.

The models are the seeded test models with a constant delta added to the EOS bias: on the unmodified no-stop run, image b emits EOS
at the first step whose margin max_{v != eos} logit_v - logit_eos is below delta, and the trajectory before that step is the same, so
the first-EOS steps of each delta are known before the timed runs.  Per delta: the mean first-EOS step, the mean over image groups of
the group's last one (what the fused kernel's exit depends on: groups of 4 = the serial launch at B = 64 on 148 SMs, 16 = the
pipeline's clusters; the per-operation chain of config T waits for the whole batch), and img/s of the serial graph-replayed
generate_tokens and of GenerationPipeline, stop off and on alternately, `--reps` times.  delta = +1e4: every image at step 0;
delta = -1e4: no image ever finishes (the cost of stopping when it never triggers).

  python tools/eos_stop_probe.py --out RESULT.json [--configs P,T] [--reps 3]
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

EOS = 301
B, T = 64, 99


def model_of(config):
    if config == "P":
        return cases.build_product_model("P", seed=0, gamma_seed=5).to("cuda").set_precision("bf16")
    cases.product_cfg(100)
    torch.manual_seed(4)
    enc = M.Encoder(model_name=cases.VIT, pretrained=False, out_dim=1024)
    m = M.EncoderDecoder(enc, M.Decoder(332, 196, 1024, 8, 8)).eval()
    g = torch.Generator().manual_seed(9)
    with torch.no_grad():
        for k, p in m.named_parameters():
            if k.endswith("gamma"):
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)
    return m.to("cuda").set_precision("bf16")


def first_eos(margin, delta):
    """(B,) first step with margin < delta, T where there is none."""
    hit = margin < delta
    return torch.where(hit.any(1), hit.float().argmax(1), torch.full((margin.shape[0],), margin.shape[1]))


def group_max_mean(e, g):
    return float(torch.stack([c.max() for c in e.split(g)]).float().mean())


def timed(fn, n):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn(n)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="P,T")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", required=True, help="JSON file for the results (GPU name and power limit included)")
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip(), "B": B, "T": T, "reps": a.reps, "configs": {}}
    print(res["gpu"], "|", res["nvidia_smi"], flush=True)
    for config in a.configs.split(","):
        m = model_of(config)
        xs = [cases.images(B, seed=1000 + i).to("cuda") for i in range(4)]
        _, _, lg = m.generate_tokens(xs[0], T, return_logits=True, use_graph=False)
        others = lg.clone()
        others[..., EOS] = -float("inf")
        margin = (others.max(-1).values - lg[..., EOS]).float().cpu()
        del lg, others
        # two deltas from the margins: mean first-EOS step near 22 (one box: BOS, 303, ~13 words, 304, 5 box tokens, EOS) and near 45
        grid = torch.quantile(margin.flatten(), torch.linspace(0.0005, 0.2, 400))
        picks = []
        for target in (22, 45):
            d = min(grid.tolist(), key=lambda d: abs(float(first_eos(margin, d).float().mean()) - target))
            picks.append(d)
        n_serial, n_pipe = (20, 40) if config == "P" else (6, 12)
        rows = []
        for delta in picks + [1e4, -1e4]:
            e = first_eos(margin, delta)
            row = {"delta": delta, "mean_first_eos_step": float(e.float().mean()), "mean_group_max_4": group_max_mean(e, 4),
                   "mean_group_max_16": group_max_mean(e, 16), "batch_max": int(e.max()), "never": int((e == T).sum()),
                   "serial_img_s": {"off": [], "on": []}, "pipeline_img_s": {"off": [], "on": []}}
            b = m.decoder.output.bias
            with torch.no_grad():
                saved = b[EOS].clone(); b[EOS] += delta
            pipes = {mode: M.GenerationPipeline(m, B, T, eos_token=(EOS if mode == "on" else None)) for mode in ("off", "on")}
            def serial(mode):
                kw = {"eos_token": EOS} if mode == "on" else {}
                def run(n):
                    for i in range(n):
                        m.generate_tokens(xs[i % len(xs)], T, **kw)
                return run
            def pipe(mode):
                def run(n):
                    for i in range(n):
                        pipes[mode].submit(xs[i % len(xs)])
                    pipes[mode].join()
                return run
            for mode in ("off", "on"):        # warm-up: plans, graphs
                serial(mode)(2); pipe(mode)(pipes[mode].depth)
            for _ in range(a.reps):
                for mode in ("off", "on"):
                    row["serial_img_s"][mode].append(n_serial * B / timed(serial(mode), n_serial))
                    row["pipeline_img_s"][mode].append(n_pipe * B / timed(pipe(mode), n_pipe))
            with torch.no_grad():
                b[EOS] = saved
            del pipes
            torch.cuda.empty_cache()
            rows.append(row)
            med = lambda v: sorted(v)[len(v) // 2]
            print(f"{config} delta={delta:+.3g}: first EOS mean {row['mean_first_eos_step']:.1f}, group max (4) {row['mean_group_max_4']:.1f}, "
                  f"(16) {row['mean_group_max_16']:.1f}, batch max {row['batch_max']}, never {row['never']} | serial img/s off "
                  f"{med(row['serial_img_s']['off']):.0f} on {med(row['serial_img_s']['on']):.0f} | pipeline off "
                  f"{med(row['pipeline_img_s']['off']):.0f} on {med(row['pipeline_img_s']['on']):.0f}", flush=True)
        res["configs"][config] = rows
        del m
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
