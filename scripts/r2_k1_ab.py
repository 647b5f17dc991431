"""K1 A/B timing on one GPU: 8 chunks of 32768 rays x 128 samples through Engine.network (CUDA events), fp16 and bf16."""
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
from oracle import cfnerf_oracle as O

dev = torch.device("cuda:0")
cfg = O.CfnConfig()
N = 128
B = 32768
rays = O.synthetic_rays(B, 1).to(dev)
res = {}
for prec in ("fp16", "bf16"):
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, O.make_params(cfg, 0), *O.make_latents(cfg, 0)).to(dev)
    eng = cf.engine_for(net, dev, prec)
    z = eng.zvals(rays, cf.reference_t_schedule(N, dev), None, False)
    for _ in range(6):
        fp = eng.network(B, N, rays=rays, z_vals=z)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(24):
        fp = eng.network(B, N, rays=rays, z_vals=z)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 24
    res[prec] = {"ms": ms, "tflops": B * N * 4708864 / ms / 1e9, "rays_per_s": B / ms * 1e3}
    # correctness against the fp32 check mode on a slice
    ref = cf.engine_for(net, dev, "fp32").network(256, N, rays=rays[:256], z_vals=z[:256])
    res[prec]["max_err_vs_fp32"] = float((fp[:256 * N] - ref).abs().max())
print(json.dumps({"lib": os.environ.get("CFN_AB_LIB", "tree"), **res}))
