"""Probe of the batch pipeline's operating point: images per decode cluster (SMs per batch) x decode streams x depth [x CTAs per SM].
usage: pipeline_probe.py [K] [ipc,streams,depth[,ctas_per_sm] ...]"""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import cases
import mdcnet_b200 as M
B, T, K = 64, 99, int(sys.argv[1]) if len(sys.argv) > 1 else 16
m = cases.build_product_model("P", seed=0, gamma_seed=5).to("cuda").set_precision("bf16")
xs = [cases.images(B, seed=100 + i).to("cuda") for i in range(4)]
for _ in range(3): m.generate_tokens(xs[0], T)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
outs = [m.generate_tokens(xs[i % 4], T)[0] for i in range(K)]
b.record(); torch.cuda.synchronize()
print(f"serial                                  : {B * K / (a.elapsed_time(b) / 1e3):9.1f} img/s  ({a.elapsed_time(b) / K:.3f} ms/batch)")
cfgs = [tuple(int(v) for v in c.split(',')) for c in sys.argv[2:]] or [(16, 4, 6, 0), (8, 4, 6, 2), (8, 5, 8, 2), (8, 6, 8, 2)]
for cfg in cfgs:
    ipc, ndec, depth = cfg[:3]; cps = cfg[3] if len(cfg) > 3 else 0
    pipe = M.GenerationPipeline(m, B, T, depth=depth, decode_streams=ndec, images_per_cluster=ipc, ctas_per_sm=cps)
    def run(K):
        res = [pipe.submit(xs[i % 4]).tokens for i in range(K)]
        pipe.join()
        return res
    run(2 * depth); torch.cuda.synchronize()
    a.record()
    res = run(K)
    b.record(); torch.cuda.synchronize()
    ok = all(torch.equal(r, o) for r, o in zip(res, outs))
    print(f"images/cluster {ipc} ctas/SM {cps} decode streams {ndec} depth {depth}: {B * K / (a.elapsed_time(b) / 1e3):9.1f} img/s  ({a.elapsed_time(b) / K:.3f} ms/batch)  equal: {ok}")
    del pipe
