#!/usr/bin/env python
"""bench.py -- images/sec of MDC-Net's batched inference hot path (encode + greedy decode) on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config 1|4|5] [--global-batch G] [--dump-outputs DIR]

--dump-outputs DIR: after the timed steps, the results of the last one (tokens, confidences; boxes and max IoU for --config 5) as
float32 DIR/<name>.npy.  Weights and inputs are seeded, so two builds run with the same arguments can be compared array for array.

A "step" = one batch of synthetic NEU-DET-shaped images (200x200 gray u8 -> the reference transform -> 3x224x224) through
encoder -> cross-K/V -> greedy decode.  Default workload = BASELINE.json configs[1]: config P, B = 64 per GPU, bf16, 99 new tokens.
N > 1 (torchrun): every rank owns its own 64 images (weak scaling; at 8 ranks this is configs[2]'s B = 512), the run ends with ONE
all-gather of all ranks' packed results (tokens + confidences of every step), inside the timed region; `--global-batch 512` runs
configs[2] as written (512 images split over the ranks, strong scaling).  `--config 4` / `--config 5` print the line for
configs[3] (512x512 inputs, 1024 memory keys) / configs[4] (256 new tokens, top-k 5 sampling, B = 256, + token->box decode + IoU inside
the timed region); the default line carries short runs of both under "other_configs" (N = 1).  Prints ONE JSON line on rank 0.

  value   : K steps through the batch pipeline (mdcnet_b200.GenerationPipeline: the encoder of step i+1 overlaps the decode loops of
            earlier steps on other streams), device-resident inputs, CUDA events around the K steps, max over ranks
  e2e     : the public streaming API generate_stream(model, pinned host batches, tokenizer, max_len): H2D of every batch and D2H of
            its results inside; e2e_gray_u8: the same from raw 200x200 u8 images (fused transform kernel on the device)
  serial  : one batch at a time (generate_tokens / generate), 256 MiB L2 flush between steps
  roofline: the dominant kernel (fused decode loop): algorithmic bytes (SURVEY 8d) of one batch / pipelined ms_per_step against the
            measured HBM peak (up to four launches of the kernel share the GPU with the encoder inside the timed region);
            `launch_alone` = the same launch (16 images per cluster, 32 SMs) timed alone with CUDA events, `serial` = the low-latency
            instantiation generate() uses, `full_gpu` = a B = 256 launch that fills the GPU with decode clusters;
            roofline_gemm: mlp.fc1 against the measured bf16 tensor peak
  cpu_baseline: the oracle port of the reference's own loop (encoder recomputed every step, model.py:177-181) on the host cores,
            bounded sample (N = 1 only); gpu_eager_baseline: the same restated algorithm as plain PyTorch eager bf16 on this GPU.
  --impl reference prints only the CPU arm (rank 0).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec end-to-end encode+greedy decode"
VIT = "deit3_medium_patch16_224.fb_in22k_ft_in1k"

# BASELINE.json configs -> workloads (bench config id = 1-based index into BASELINE.json `configs`, minus the CPU-only configs[0])
WORKLOADS = {
    1: dict(name="configs[1]", img=224, S=196, B=64, T=99, top_k=0, max_len=100,
            text="MDC-Net config P (deit3_medium 224 + 6-layer dim-256 decoder, V=305), batch 64/GPU, 99 greedy tokens, synthetic 200x200 gray -> 3x224x224"),
    4: dict(name="configs[3]", img=512, S=1024, B=128, T=99, top_k=0, max_len=100,
            text="encoder stress: 512x512 inputs (32x32 = 1024 patches: 5.2x the memory of 224; BASELINE's '4x' would be 448), batch 128, "
                 "1025-token encoder strips, cross-attention over 1024 memory keys, 99 greedy tokens"),
    5: dict(name="configs[4]", img=224, S=196, B=256, T=256, top_k=5, max_len=257,
            text="long decode: 256 new tokens, top-k 5 sampling (seeded uniforms), batch 256, paged KV cache (17 pages of 16 tokens per image), "
                 "then token->box decode and batched max-IoU against synthetic ground truth, all inside the timed region"),
    # not a BASELINE.json config: the geometry the reference was TRAINED with (trail_01.py:158-160), outside the fused decode kernel's shape
    6: dict(name="geometry T", img=224, S=196, B=64, T=99, top_k=0, max_len=100, dim=1024, heads=8, layers=8, vocab=332,
            text="trained geometry (trail_01.py:158-160): deit3_medium 224 + 8-layer dim-1024 decoder (8 heads x 128, FFN 2048, V=332), batch 64, "
                 "99 greedy tokens; decode = the per-operation chain (weight-streaming tensor-core linears, key-split cross-attention), 8 decode streams"),
}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """SM clock + throttle reasons DURING the timed region (B200_PROFILING.md recipe), sampled every 10 ms through NVML in a
    background thread (nvidia-smi -lms needs ~0.5 s to start, longer than a short timed region); nvidia-smi is the fallback."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.samples, self.run, self.t, self.h, self.mx = index, [], False, None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def _loop(self):
        nv = self.nv
        while self.run:
            try:
                self.samples.append((float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)), int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))))
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        self.samples = []
        if self.h is not None:
            self.run = True
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()

    def stop(self):
        if self.h is None:
            return self._smi_once()
        self.run = False
        self.t.join(timeout=1.0)
        sm = [c for c, _ in self.samples]
        mask = 0
        for _, r in self.samples:
            mask |= r
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.mx, "reasons": [n for b, n in self.REASONS.items() if mask & b],
                "samples": len(sm), "source": "nvml, 10 ms period"}

    def _smi_once(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            r = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10)
            c = [x.strip() for x in r.stdout.strip().split(",")]
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            return {"sm_mhz": float(c[0]), "sm_max_mhz": float(c[1]), "reasons": [n for i, n in enumerate(names) if c[2 + i].lower().startswith("active")],
                    "samples": 1, "source": "nvidia-smi, one sample right after the timed region (NVML unavailable)"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}


# ---- synthetic workload (no oracle import on the GPU arm) --------------------------------------------------------------------
def synth_gray_u8(B, hw=200, seed=1234):
    """NEU-DET-shaped synthetic images: u8 (B, hw, hw), seeded."""
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (B, hw, hw), generator=g, dtype=torch.uint8)


def build_model(M, img=224, S=196, max_len=100, seed=0, gamma_seed=5, dim=256, heads=8, layers=6, vocab=305):
    """Random-init MDC-Net config P through the product constructors (inference_p.py:126-129: dim 256, 8 heads, 6 layers, V = 305),
    LayerScale gammas redrawn from U(0.5, 1.5) (random-init DeiT-III has gamma = 1e-6, which would make the encoder a no-op)."""
    M.CFG.max_len, M.CFG.pad_idx, M.CFG.bos_idx = max_len, 302, 300
    torch.manual_seed(seed)
    enc = M.Encoder(model_name=VIT, pretrained=False, out_dim=dim, img_size=img)
    dec = M.Decoder(vocab, S, dim, heads, layers)
    model = M.EncoderDecoder(enc, dec)
    g = torch.Generator().manual_seed(gamma_seed)
    with torch.no_grad():
        for k, p in model.named_parameters():
            if k.endswith("gamma"):
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)
    return model.eval()


# ---- CPU reference arm ------------------------------------------------------------------------------------------------------
def cpu_reference_arm(timed_iters, warmup_iters, sample_steps=6, T=99, batches=(1, 8)):
    """The reference's own CPU path, restated (oracle port): the generate() loop of inference_p.py:69-90 with the encoder recomputed
    every step (model.py:177-181, Q9), fp32, all host threads.  Bounded sample: `sample_steps` of the T decode steps at B = 1 and
    B = 8, extrapolated linearly to T.  The port's decoder runs over the PREFIX only (causally equivalent to the reference's
    PAD-padded full-length pass, and cheaper: the reported number flatters the CPU)."""
    from oracle import cases, mdc_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model = cases.build_product_model("P", seed=0, gamma_seed=5)
    sd, cfg = cases.state_dict_of(model), cases.oracle_cfg("P")
    detail, best, best_iter_s = {}, None, None
    with torch.no_grad():
        for B in batches:
            x = cases.images(B)
            times = []
            for i in range(warmup_iters + timed_iters):
                t0 = time.perf_counter()
                O.generate(sd, x, cfg, max_len=sample_steps, recompute_encoder=True)
                dt = time.perf_counter() - t0
                if i >= warmup_iters:
                    times.append(dt)
            per_step = statistics.mean(times) / sample_steps
            img_s = B / (per_step * T)
            detail[f"B={B}"] = {"images_per_s": img_s, "ms_per_token": per_step * 1e3, "iterations_timed": len(times)}
            if best is None or img_s > best:
                best, best_iter_s = img_s, statistics.mean(times)
    return {"value": best, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": f"oracle port of the reference generate() loop (encoder recomputed each step, prefix-only decoder), {sample_steps} of {T} decode "
                      f"steps extrapolated x{T}/{sample_steps}, measured at B = {' and '.join(str(b) for b in batches)} ({timed_iters} timed + {warmup_iters} warm-up "
                      f"iterations each); value = the better of the two", "detail": detail}, best_iter_s


def gpu_eager_baseline(dev, B=8, sample_steps=6, T=99):
    """The same restated algorithm (reference loop, encoder recomputed per step) as plain PyTorch eager kernels in bf16 on THIS GPU:
    the 'existing library kernels' bar next to the CPU number.  Bounded sample, extrapolated like the CPU arm."""
    try:
        from oracle import cases, mdc_oracle as O
        model = cases.build_product_model("P", seed=0, gamma_seed=5)
        sd = {k: (v.to(dev, torch.bfloat16) if v.is_floating_point() else v.to(dev)) for k, v in cases.state_dict_of(model).items()}
        cfg = cases.oracle_cfg("P")
        x = cases.images(B).to(dev, torch.bfloat16)
        with torch.no_grad():
            O.generate(sd, x, cfg, max_len=2, recompute_encoder=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            O.generate(sd, x, cfg, max_len=sample_steps, recompute_encoder=True)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
        per_step = dt / sample_steps
        return {"value": B / (per_step * T), "unit": "images/s", "kind": "port (oracle restatement on torch CUDA eager kernels, bf16)",
                "sample": f"B = {B}, {sample_steps} of {T} steps of the reference loop (encoder recomputed each step), extrapolated; {per_step * 1e3:.1f} ms/token"}
    except Exception as e:      # a reported baseline must never take the bench line down
        return {"value": None, "error": f"{type(e).__name__}: {e}"[:300]}


# ---- roofline helpers ---------------------------------------------------------------------------------------------------------
def decode_algorithmic_bytes(B, T, S, dim=256, layers=6, ffn=2048, vocab=305):
    """SURVEY 8(d) / DESIGN.md: bytes one decode launch (T steps) must move, bf16 storage:
    per step  B*(cross_KV + self_KV(t)) + W_step + B*(V*4 + 2*dim*2)."""
    cross = layers * 2 * S * dim * 2                                   # 1 204 224 B / image at S = 196
    w_step = layers * (3 * dim * dim + 3 * dim * dim + 2 * dim * ffn) * 2 + vocab * dim * 2   # decode-touched weights
    per_step_fixed = B * cross + w_step + B * (vocab * 4 + 2 * dim * 2)
    self_kv = sum(B * layers * 2 * t * dim * 2 for t in range(T))
    return T * per_step_fixed + self_kv


def ncu_traffic(name):
    """DRAM bytes per launch of `name` from the newest committed ncu --set full capture (profiles/*_traffic.json), or None."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
    if not files:
        return None
    try:
        return json.load(open(files[-1])).get(name, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def decode_launch_ms(model, x_dev, dev, T, ipc, top_k=0, reps=3, cps=0):
    """One decode launch (T steps, B images) timed alone with CUDA events on the launching stream."""
    eng = model._engine(dev)
    _, memory = eng.encode(x_dev, want_enc_out=False, want_memory=True)
    ckv = eng.cross_kv(memory)
    Bn = x_dev.shape[0]
    tokens = torch.full((Bn, T + 1), 302, dtype=torch.int32, device=dev); tokens[:, 0] = 300
    uni = torch.rand((Bn, T), device=dev) if top_k else None
    kv, scratch = eng.decode(ckv, tokens, 0, T, max_tokens=T, forced=False, images_per_cluster=ipc, ctas_per_sm=cps, top_k=top_k, uniforms=uni)
    torch.cuda.synchronize()
    best = None
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.decode(ckv, tokens, 0, T, max_tokens=T, forced=False, kv=kv, scratch=scratch, images_per_cluster=ipc, ctas_per_sm=cps, top_k=top_k, uniforms=uni)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        best = ms if best is None else min(best, ms)
    return best


def decode_roofline(model, x_dev, dev, peaks, T, S, ipc, top_k=0, cps=0, geo=None):
    B = x_dev.shape[0]
    ms = decode_launch_ms(model, x_dev, dev, T, ipc, top_k, cps=cps)
    if geo:                                             # a geometry outside the fused kernel: the per-operation chain, one batch alone
        nbytes = decode_algorithmic_bytes(B, T, S, dim=geo["dim"], layers=geo["layers"], ffn=2048, vocab=geo["vocab"])
        ach = nbytes / (ms / 1e3) / 1e9
        return {"kernel": f"per-operation decode chain (prep_x_half / dec_linear_stream / dec_self_attn / dec_cross_attn_split / dec_select kernels, "
                          f"{11 * geo['layers'] + 3} launches per token), one batch alone, eager launches; {T} decode steps x {geo['layers']} layers, B={B}, S={S}",
                "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": None,
                "algorithmic_bytes_per_launch": nbytes, "ms_per_launch": ms, "ms_per_decode_token": ms / T,
                "peak_src": peaks["src"] + " HBM copy bandwidth (chain timed alone, CUDA events)"}
    nbytes = decode_algorithmic_bytes(B, T, S)
    ach = nbytes / (ms / 1e3) / 1e9
    n_cl = -(-B // (16 if ipc > 8 else (ipc or 5)))
    inst = (f"16 images per 8-CTA cluster, two column blocks per pass (the instantiation the batch pipeline runs): {n_cl} clusters = {8 * n_cl} of 148 SMs" if ipc > 8 else
            (f"compact layout, 8 images per cluster, two clusters per SM: {n_cl} clusters on {4 * n_cl} SMs" if cps == 2 else
             "spread over as many clusters as fit, one CTA per SM (the low-latency instantiation generate() runs)"))
    return {"kernel": f"decode_fused_kernel, {inst}; one launch = {T} decode steps x 6 layers, B={B}, S={S}", "bound": "hbm", "achieved": ach,
            "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": ncu_traffic("decode16" if ipc > 8 else "decode"),
            "algorithmic_bytes_per_launch": nbytes, "ms_per_launch": ms, "ms_per_decode_token": ms / T,
            "peak_src": peaks["src"] + " HBM copy bandwidth (kernel timed alone, CUDA events)"}


def roofline_probe(M, dev, peaks, B):
    """Times the encoder's largest GEMM (mlp.fc1: M=B*197, N=2048, K=512, bias+GELU epilogue) alone."""
    L = M._lib
    Mr, N, K = B * 197, 2048, 512
    A = (torch.randn(Mr, K, device=dev) * 0.5).to(torch.bfloat16)
    W = (torch.randn(N, K, device=dev) * 0.05).to(torch.bfloat16)
    bias = torch.zeros(N, device=dev)
    D = torch.empty(Mr, N, dtype=torch.bfloat16, device=dev)

    def run():
        L.check(L.lib().mdc_gemm(L.ctx(dev), L.MDC_BF16, L.EPI_BIAS_GELU, L.ptr(A), K, L.ptr(W), K, L.ptr(D), N, L.ptr(bias), None, 0,
                                 Mr, N, K, L.stream_ptr()))
    for _ in range(5):
        run()
    torch.cuda.synchronize()
    # replayed from a CUDA graph, as the encoder phase launches it: back-to-back eager launches of a ~25 us kernel are bound by
    # the host's launch rate (~16 us floor per launch measured), which understated this kernel by 20 %
    reps, replays = 20, 5
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            run()
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(replays):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / (reps * replays)
    flops = 2.0 * Mr * N * K
    ach = flops / (ms / 1e3) / 1e12
    return {"kernel": "gemm_tc_kernel (mlp.fc1 shape, bias+GELU)", "bound": "tensor", "achieved": ach, "peak": peaks["bf16_tflops"],
            "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops"], "traffic": ncu_traffic("gemm_fc1"), "peak_src": peaks["src"] + " burst (kernel timed alone, CUDA events around CUDA-graph replays of 20 launches)",
            "ms_per_launch": ms}


# ---- one workload through the batch pipeline ------------------------------------------------------------------------------------
PIPE_KW = {}          # --decode-streams / --depth: GenerationPipeline operating point (defaults: 4 streams, 6 plans)


def dump_outputs(M, d, last, T1, C, NB):
    """Writes one step's packed results (every rank's rows) as float32 arrays DIR/<name>.npy: the tokens and confidences a caller of
    the batch pipeline receives, and for the box workload the decoded boxes and their max IoU against the ground truth."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    tokens, confs, boxes, max_iou = M.parallel.unpack_results(last, T1, C, NB)
    arrays = {"tokens": tokens, "confidences": confs, "boxes": boxes, "max_iou": max_iou}
    for name, a in arrays.items():
        if a is not None:
            np.save(os.path.join(d, name + ".npy"), a.cpu().to(torch.float32).numpy())     # token ids < 2^24: exact in float32


def run_workload(M, wl, B, steps, warmup, dev, rank, world, dist, peaks, full, dump=None):
    """Returns the fields of one bench line for workload `wl` at per-rank batch B.  full: also serial / e2e / roofline extras.
    dump: directory for the results of the last timed step (dump_outputs)."""
    T, S, img, top_k = wl["T"], wl["S"], wl["img"], wl["top_k"]
    geo = {k: wl[k] for k in ("dim", "heads", "layers", "vocab") if k in wl}
    model = build_model(M, img=img, S=S, max_len=wl["max_len"], **geo).to(dev).set_precision("bf16")
    tok = M.Tokenizer(num_bins=224, width=img, height=img, max_len=wl["max_len"])
    NROT = 4                                         # rotating input batches (4 x 38.5 MB > the 126 MB L2 at the default shape)
    gs_host = [synth_gray_u8(B, seed=4321 + 17 * rank + i).pin_memory() for i in range(NROT)]
    xs_dev = [M.preprocess_gray(g.to(dev), size=img) for g in gs_host]          # the reference transform, on the device
    xs_host = [x.cpu().pin_memory() for x in xs_dev]
    T1, C = T + 1, (T + 3) // 4
    sampling = top_k != 0
    unis = [torch.rand((B, T), generator=torch.Generator().manual_seed(77 + i)).to(dev) for i in range(NROT)] if sampling else None
    with_boxes = wl["name"] == "configs[4]"
    gt = None
    if with_boxes:                                   # synthetic ground truth (SURVEY 8d config 5): (B, 5, 4) xyxy with pad_sequence-style zero rows
        gg = torch.Generator().manual_seed(9)
        gt = torch.rand(B, 5, 4, generator=gg) * 160
        gt[..., 2:] = gt[..., :2] + 8 + torch.rand(B, 5, 2, generator=gg) * 56
        gt[torch.rand(B, 5, generator=gg) < 0.3] = 0
        gt = gt.to(dev)
    pipe = M.GenerationPipeline(model, B, T, top_k=top_k, **PIPE_KW)
    NB = max(1, (T1 + 4) // 5) if with_boxes else 0          # box slots per image (Tokenizer.decode_bboxes_padded)
    F = T1 + C + 5 * NB

    def steps_pipelined(k, sink):
        """k steps through the batch pipeline; every step packs its results (tokens, confidences[, boxes + max IoU]) into its rows of
        `sink` on its own decode stream; ONE all-gather of the whole buffer after the last step."""
        for i in range(k):
            t = pipe.submit(xs_dev[i % NROT], uniforms=unis[i % NROT] if sampling else None)
            with torch.cuda.stream(t.stream):
                if with_boxes:
                    boxes, _ = tok.decode_bboxes_padded(t.tokens)                                   # token scan kernel, no host sync
                    _, mx = M.iou._batched(M._lib.IOU_EPS, boxes, gt, want_iou=False, want_max=True)   # calculate_batch_max_iou's kernel, device result
                    sink[i * B:(i + 1) * B] = M.parallel.pack_results(t.tokens, t.confs, boxes, mx)
                else:
                    sink[i * B:(i + 1) * B] = M.parallel.pack_results(t.tokens, t.confs)
        pipe.join()
        pre = torch.cuda.Event(enable_timing=True)
        pre.record()                                 # this rank's own work is enqueued behind this point; the gather follows
        steps_pipelined.pre_gather = pre
        return M.parallel.all_gather_results(sink, k * B * world)

    sink_w = torch.zeros((max(8, warmup) * B, F), dtype=torch.int32, device=dev)
    steps_pipelined(max(8, warmup), sink_w)
    torch.cuda.synchronize()
    sink = torch.zeros((steps * B, F), dtype=torch.int32, device=dev)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(dev.index)
    sampler.start()
    n0 = M._lib.launch_count(dev)
    pa, pb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pa.record()
    out = steps_pipelined(steps, sink)
    pb.record()
    torch.cuda.synchronize()
    n1 = M._lib.launch_count(dev)
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    if dump and rank == 0:                           # rows of the gathered buffer: rank-major, then step, then image
        dump_outputs(M, dump, out.view(world, steps, B, F)[:, -1].reshape(world * B, F), T1, C, NB)
    t = torch.tensor([pa.elapsed_time(pb)], dtype=torch.float64, device=dev)
    mine = torch.tensor([pa.elapsed_time(pb), pa.elapsed_time(steps_pipelined.pre_gather)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = t.item()
    res = {"value": B * world * steps / (total_ms / 1e3), "ms_per_step": total_ms / steps, "clocks": clocks, "gpu_launches": int(n1 - n0),
           "gathered_rows": int(out.shape[0])}
    if world > 1:
        # where an N-GPU run loses against N independent GPUs: every rank's own time to finish its steps (before the gather) and its
        # time including the one all-gather -- the gather completes when the SLOWEST rank arrives, so (max - own) is waiting, not work
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        res["per_rank_ms"] = {"own_steps": [round(v[1].item(), 3) for v in allr], "with_gather": [round(v[0].item(), 3) for v in allr]}

    # end-to-end through the public streaming API (generate_stream), HOST buffers: H2D of every batch + D2H of its results inside
    def e2e_run(batches_host, k):
        n = 0
        for bp, cf in M.generate_stream(model, (batches_host[i % NROT] for i in range(k)), tok, max_len=T, top_k=top_k):
            n += bp.shape[0]
        return n

    def timed_e2e(batches_host):
        e2e_run(batches_host, 8)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        e2e_run(batches_host, steps)
        torch.cuda.synchronize()
        tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return B * world * steps / tt.item()

    res["e2e"] = {"value": timed_e2e(xs_host), "unit": "images/s", "h2d_bytes_per_step": xs_host[0].numel() * 4, "d2h_bytes_per_step": B * (T1 * 4 + C * 4)}
    if not full:
        if rank == 0:
            res["roofline"] = decode_roofline(model, xs_dev[0], dev, peaks, T, S, 16, top_k, geo=geo)
        return res, model, xs_dev
    res["e2e_gray_u8"] = {"value": timed_e2e(gs_host), "unit": "images/s", "h2d_bytes_per_step": B * 200 * 200, "d2h_bytes_per_step": B * (T1 * 4 + C * 4),
                          "note": "generate_stream over raw u8 200x200 host images; the reference transform (cv2-exact uint8 resize + normalise) runs on the device"}

    # serial: one batch at a time (generate_tokens / generate), 256 MiB L2 flush between steps (untimed)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for _ in range(3):
        model.generate_tokens(xs_dev[0], T)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(min(steps, 20))]
    for i, (a, b) in enumerate(ev):
        flush.fill_(1)
        a.record()
        model.generate_tokens(xs_dev[i % NROT], T)
        b.record()
    torch.cuda.synchronize()
    serial_ms = sum(a.elapsed_time(b) for a, b in ev) / len(ev)
    t0 = time.perf_counter()
    for i in range(len(ev)):
        M.generate(model, xs_host[i % NROT], tok, max_len=T)
    torch.cuda.synchronize()
    res["serial"] = {"value": B / (serial_ms / 1e3), "ms_per_step": serial_ms, "e2e": B * len(ev) / (time.perf_counter() - t0), "steps": len(ev),
                     "note": "per rank, one batch at a time (generate_tokens / generate), 256 MiB L2 flush between steps (untimed)"}
    return res, model, xs_dev


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--decode-streams", type=int, default=0)
    ap.add_argument("--depth", type=int, default=0)
    # default 100 steps (~0.5 s pipelined: the fill and drain of the 6-deep pipeline, ~8 ms, stay below 2 %) for config 1, 20 for the others
    ap.add_argument("--steps", type=int, default=None, help="timed steps (batches) of the workload")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=[1, 4, 5, 6], help="1: BASELINE configs[1] (default; configs[2] under torchrun), 4: configs[3], 5: configs[4], 6: the trained geometry (dim 1024)")
    ap.add_argument("--global-batch", type=int, default=0, help="total images per step, split over the ranks (configs[2]: 512); default 64 per rank")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--profile", action="store_true", help="1 warm-up + 1 serial step only (for an ncu launch list)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 100 if args.config == 1 else 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.profile):
        ap.error("--dump-outputs writes the results of the batch pipeline: not with --impl reference or --profile")
    if args.decode_streams:
        PIPE_KW["decode_streams"] = args.decode_streams
    if args.depth:
        PIPE_KW["depth"] = args.depth
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    wl = WORKLOADS[args.config]
    B = wl["B"]
    scaling = "weak"
    if args.global_batch:
        assert args.global_batch % world == 0, "--global-batch must divide evenly over the ranks"
        B, scaling = args.global_batch // world, "strong"
    cfg = {"workload": (f"BASELINE {wl['name']}: " if args.config != 6 else "") + wl["text"], "global_batch": B * world, "batch_per_gpu": B, "new_tokens": wl["T"],
           "parallelism": f"dp{world}", "sampler": "greedy" if not wl["top_k"] else f"top-k {wl['top_k']} (seeded uniforms)",
           "pipeline": ("batch pipeline (GenerationPipeline / generate_stream): 6 plans, 4 decode streams at 16 images per 8-CTA cluster + 1 encoder stream; steps overlap, every step does all of its work inside the timed region"
                        if args.config != 6 else "batch pipeline (GenerationPipeline / generate_stream): 10 plans, 8 decode streams (per-operation decode graphs) + 1 encoder stream"),
           "collective": "ONE all-gather of every rank's packed results (all steps) at the end of the timed region; none inside the decode loop",
           "l2": "no flush inside the pipelined region: 4 rotating input batches and a per-step working set (activations, cross-K/V, KV pages) well above the 126 MB L2"}

    if args.impl == "reference":
        if rank != 0:
            return
        timed = max(1, min(args.steps, 3)); warm = min(max(args.warmup, 0), 1)
        base, iter_s = cpu_reference_arm(timed, warm)
        out = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "images/s", "n_gpus": args.gpus, "steps": timed, "warmup": warm,
               "steps_requested": args.steps, "warmup_requested": args.warmup,
               "ms_per_step": iter_s * 1e3, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
               "dtype": "f32", "data": "synthetic", "config": cfg, "cpu_baseline": base,
               "note": "each timed 'step' is one bounded sample of the workload (6 of 99 decode steps of the reference loop at B = 1 and at B = 8), not a full 64-image batch: see cpu_baseline.sample",
               "e2e": {"value": base["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(out))
        return

    import torch.distributed as dist
    import mdcnet_b200 as M
    assert torch.cuda.is_available(), "bench.py needs a B200"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()

    if args.profile:
        model = build_model(M).to(dev).set_precision("bf16")
        x = M.preprocess_gray(synth_gray_u8(64).to(dev))
        model.generate_tokens(x, 99); torch.cuda.synchronize()
        n0 = M._lib.launch_count(dev)
        model.generate_tokens(x, 99); torch.cuda.synchronize()
        print(json.dumps({"profile_step_launches": int(M._lib.launch_count(dev) - n0)}))
        return

    steps = args.steps
    res, model, xs_dev = run_workload(M, wl, B, steps, args.warmup, dev, rank, world, dist, peaks, full=(args.config == 1), dump=args.dump_outputs)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    out = {"metric": METRIC, "value": res["value"], "unit": "images/s", "n_gpus": world, "steps": steps, "warmup": max(8, args.warmup),
           "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "bf16",
           "data": "synthetic", "config": cfg, "clocks": res["clocks"], "e2e": res["e2e"], "gpu_launches": res["gpu_launches"]}
    if "per_rank_ms" in res:
        out["per_rank_ms"] = res["per_rank_ms"]
    if args.config == 1:
        # The dominant kernel is the fused decode loop.  In the timed region four of its launches (32 SMs each) and the encoder share the
        # GPU, so the figure that belongs to the headline is the rate at which the decode loops TOGETHER move their algorithmic bytes:
        # bytes of one batch / pipelined ms_per_step.  Beside it: the same launch timed alone (a 32-SM launch: its fraction of the
        # whole GPU's HBM peak says how small a slice of the GPU one batch is given), the low-latency instantiation generate() runs,
        # and a launch that fills the GPU with decode clusters (B = 256, two clusters per SM).
        alone = decode_roofline(model, xs_dev[0], dev, peaks, wl["T"], wl["S"], 16)
        nbytes = alone["algorithmic_bytes_per_launch"]
        ach = nbytes / (res["ms_per_step"] / 1e3) / 1e9
        roof = {"kernel": "decode_fused_kernel (one launch = 99 decode steps x 6 layers of one 64-image batch; 16 images per 8-CTA cluster) as the "
                          "timed region runs it: up to four launches in flight next to the encoder of the following batches",
                "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": alone["traffic"],
                "algorithmic_bytes_per_launch": nbytes, "ms_per_launch": res["ms_per_step"],
                "how": "algorithmic decode bytes of one batch (SURVEY 8d: cross-K/V + self-K/V + decode-touched weights + logits, 11.28 GB) / pipelined "
                       "ms_per_step; CUDA events around the timed region; `traffic` = DRAM bytes of one launch from the committed ncu capture",
                "peak_src": peaks["src"] + " HBM copy bandwidth",
                "launch_alone": alone,
                "serial": decode_roofline(model, xs_dev[0], dev, peaks, wl["T"], wl["S"], 0)}
        x256 = torch.cat([xs_dev[i % len(xs_dev)] for i in range(4)], dim=0)
        roof["full_gpu"] = decode_roofline(model, x256, dev, peaks, wl["T"], wl["S"], 8, cps=2)
        del x256
        roof["ms_per_decode_token"] = alone["ms_per_decode_token"]
        out.update({"ms_per_decode_token": roof["ms_per_decode_token"], "roofline": roof, "roofline_gemm": roofline_probe(M, dev, peaks, B),
                    "e2e_gray_u8": res["e2e_gray_u8"], "serial": res["serial"]})
        del model
        if world == 1 and not args.no_other_configs:       # short runs of configs[3] / configs[4] so that their lines are in the record
            other = {}
            for cid in (4, 5, 6):
                w2 = WORKLOADS[cid]
                n2 = 16 if cid == 6 else 6      # geometry T runs 10 plans deep: a 6-step run is mostly fill and drain
                try:
                    r2, m2, _ = run_workload(M, w2, w2["B"], n2, 3, dev, rank, world, dist, peaks, full=False)
                    other[w2["name"]] = {"workload": w2["text"], "batch": w2["B"], "new_tokens": w2["T"], "steps": n2, "value": r2["value"], "unit": "images/s",
                                         "ms_per_step": r2["ms_per_step"], "e2e": r2["e2e"], "roofline": r2["roofline"], "gpu_launches": r2["gpu_launches"]}
                    del m2
                except Exception as e:
                    other[w2["name"]] = {"error": f"{type(e).__name__}: {e}"[:300]}
                torch.cuda.empty_cache()
            out["other_configs"] = other
        if world == 1 and not args.no_cpu_baseline:          # reported on rank 0 at N = 1 only; `--impl reference` is the arm for every N
            out["cpu_baseline"], _ = cpu_reference_arm(1, 1)
            out["gpu_eager_baseline"] = gpu_eager_baseline(dev)
    else:
        out["roofline"] = res["roofline"]
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
