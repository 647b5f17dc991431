"""What gradients with respect to the rays (F7) cost on one GPU.

On the africa architecture (8x512, F = 4, K = 32) with `default`-variant weights, one training step = render_rays
(train mode) + trainer_loss + backward, timed with a host clock around the step ending in a device synchronise (median of
--reps after --warmup), for:
  rays 512 / 4096  x  chain bf16 / tf32  x  ray gradient off / on (ray_batch.requires_grad)
and one pose-refinement step: rays_from_pose (64 x 64 image, requires_grad pose) + render_rays (test mode, tf32 chain)
+ MSE + backward with the network frozen (no weight gradients: cfn_network_bwd_inputs with grads = NULL).

Writes profiles/r06_raygrad_bench.json (or --out) with the card's name, power limit and max SM clock.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import cfnerf_oracle as O          # noqa: E402


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()
    return {"query": q[0], "value": q[1] if len(q) > 1 else ""}


def median_ms(fn, warmup: int, reps: int) -> float:
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_raygrad_bench.json"))
    a = ap.parse_args()
    import cfnerf_b200 as cf
    dev = torch.device("cuda:0")
    cfg = O.CfnConfig()
    p = O.make_params(cfg, 0, "default")
    sa, sr = O.make_latents(cfg, 0)
    res = {"gpu": gpu_info(), "config": "africa 8x512 F=4 K=32", "reps": a.reps, "warmup": a.warmup, "train_step_ms": {}}
    g = torch.Generator().manual_seed(0)
    for B in (512, 4096):
        rays = O.synthetic_rays(B, 1).to(dev)
        target = torch.rand(B, 3, generator=g).to(dev)
        t_rand = torch.rand(B, 128, generator=g).to(dev)
        for prec in ("bf16", "tf32"):
            net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev)
            for rg in (False, True):
                def step():
                    net.zero_grad(set_to_none=True)
                    r = rays.detach().requires_grad_(rg)
                    out = cf.render_rays(r, net, None, 128, True, False, perturb=1., t_rand=t_rand, precision=prec)
                    cf.trainer_loss(out, target, cfg.K)["loss"].backward()
                ms = median_ms(step, a.warmup, a.reps)
                res["train_step_ms"][f"B{B}_{prec}_raygrad{int(rg)}"] = ms
                print(f"train step B={B} {prec} ray-grad={rg}: {ms:.3f} ms", flush=True)
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev).requires_grad_(False)
    H = W = 64
    pose0 = torch.tensor([[1., 0, 0, 0.1], [0, 1, 0, -0.1], [0, 0, 1, 4.0]], device=dev)
    target = torch.rand(H * W, 3, device=dev)

    def pose_step():
        pose = pose0.clone().requires_grad_(True)
        rays = cf.rays_from_pose(H, W, 60.0, pose, 2., 6.)
        rgb = cf.render_rays(rays, net, None, 128, False, False, precision="tf32")["rgb_map"].mean(-1)
        ((rgb - target) ** 2).mean().backward()
    ms = median_ms(pose_step, a.warmup, a.reps)
    res["pose_step_ms"] = {"rays": H * W, "chain": "tf32", "frozen_network": True, "ms": ms}
    print(f"pose-refinement step ({H * W} rays, tf32, frozen network): {ms:.3f} ms", flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
