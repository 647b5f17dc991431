"""Round-2 training micro-benchmarks on one GPU (CUDA events): K2 (train flavour) and K4 alone at 4096 rays, and the whole
FusedTrainStep at 512 / 4096 rays, eager vs CUDA-graph replay.  Writes gpurun_out/r2_train_bench.json."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

import cfnerf_b200 as cf
if os.environ.get("CFN_AB_LIB"):   # same-box A/B against another build of the library
    import cfnerf_b200._lib as _L
    _L.LIB_PATH = os.environ["CFN_AB_LIB"]
from cfnerf_b200 import dist as D
from oracle import cfnerf_oracle as O

dev = torch.device("cuda:0")
cfg = O.CfnConfig()
N, K = 128, cfg.K
PREC = os.environ.get("CFN_TRAIN_PRECISION", "bf16")


def timeit(fn, iters=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


res = {}
net = cf.NeRFFlowsParams.from_oracle_params(cfg, O.make_params(cfg, 0, "lively"), *O.make_latents(cfg, 0)).to(dev)
eng = cf.engine_for(net, dev, PREC)
for B in (512, 4096):
    rays = O.synthetic_rays(B, 1).to(dev)
    z = eng.zvals(rays, cf.reference_t_schedule(N, dev), torch.rand(B, N, device=dev), False)
    fp = eng.network(B, N, rays=rays, z_vals=z, save=False) if PREC != "fp32" else eng.network(B, N, rays=rays, z_vals=z)
    ea, er = torch.randn(K, device=dev), torch.randn(K, 3, device=dev)
    out = eng.flow_composite(fp, z, rays[:, 3:6], 11, ea, er, False, train=True, want_trans=True)
    g_rgb = torch.randn(B, 3, K, device=dev) * 1e-3
    g_ld = torch.full((B, 2), -0.01 / (B * N * K), device=dev)
    res[f"k2_train_fwd_ms_{B}"] = timeit(lambda: eng.flow_composite(fp, z, rays[:, 3:6], 11, ea, er, False, train=True, want_trans=True))
    res[f"k4_bwd_ms_{B}"] = timeit(lambda: eng.flow_composite_bwd(fp, z, rays[:, 3:6], 11, ea, er, False, g_rgb, None, g_ld, trans=out["trans"], seg_sums=out["seg_sums"]))
    print(json.dumps({k: v for k, v in res.items() if k.endswith(str(B))}), flush=True)

g = torch.Generator().manual_seed(2)
for B in (512, 4096):
    for graph in (False, True):
        net = cf.NeRFFlowsParams.from_oracle_params(cfg, O.make_params(cfg, 0), *O.make_latents(cfg, 0)).to(dev)
        tr = D.FusedTrainStep(net, lr=5e-4, precision=PREC, use_graph=graph)
        rays = O.synthetic_rays(B, 1).to(dev)
        target = torch.rand(B, 3, generator=g).to(dev)
        ms = timeit(lambda: tr.step(rays, target, want_loss=False), iters=20, warm=4)
        l = tr.step(rays, target)
        res[f"train_step_ms_{B}_{'graph' if graph else 'eager'}"] = ms
        print(json.dumps({"rays": B, "graph": graph, "ms": ms, "rays_per_s": B / ms * 1e3, "loss": float(l["loss"])}), flush=True)
        del tr, net
        torch.cuda.empty_cache()
# depth-supervised step of the shipped recipe: 512 colour rays + 128 depth rays
net = cf.NeRFFlowsParams.from_oracle_params(cfg, O.make_params(cfg, 0), *O.make_latents(cfg, 0)).to(dev)
tr = D.FusedTrainStep(net, lr=5e-4, precision=PREC, use_graph=True, depth_lambda=0.01)
rays, drays = O.synthetic_rays(512, 1).to(dev), O.synthetic_rays(128, 2).to(dev)
target, td = torch.rand(512, 3, generator=g).to(dev), (1.2 + 6.8 * torch.rand(128, generator=g)).to(dev)
ms = timeit(lambda: tr.step(rays, target, want_loss=False, depth_rays=drays, target_depth=td), iters=20, warm=4)
res["train_step_ms_512+128depth_graph"] = ms
print(json.dumps({"rays": "512+128 depth", "graph": True, "ms": ms}), flush=True)
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
json.dump(res, open(os.path.join(ROOT, "gpurun_out", "r2_train_bench.json"), "w"), indent=1)
