"""What gradients with respect to the rays (F7) cost on one GPU.

On the africa architecture (8x512, F = 4, K = 32) with `default`-variant weights, one training step = render_rays
(train mode) + trainer_loss + backward, timed with a host clock around the step ending in a device synchronise (median of
--reps after --warmup), for:
  rays 512 / 4096  x  chain bf16 / tf32  x  ray gradient off / on (ray_batch.requires_grad)
and one pose-refinement step: rays_from_pose (64 x 64 image, requires_grad pose) + render_rays (test mode, tf32 chain)
+ MSE + backward with the network frozen (no weight gradients: cfn_network_bwd_inputs with grads = NULL).

Writes profiles/r06_raygrad_bench.json (or --out) with the card's name, power limit and max SM clock.

--config fern: the coarse+fine leg (render_rays(..., detach_z_samples=True)) on fern's architecture: 8x512, F = 4, K = 64,
two networks, NDC rays of a 1008 x 756 pose, 64 coarse + 128 resampled samples per ray.  One training step = render_rays
(train mode) + trainer_loss on the fine and on the coarse maps + backward, for
  rays 1024 / 4096  x  chain bf16 / tf32  x  ray gradient off / on
and one localisation step: rays_from_pose (756 x 1008, requires_grad pose) -> a fixed subsample of 4096 pixels ->
coarse+fine render_rays (test mode, tf32 chain) + MSE + backward with both networks frozen.  Writes
profiles/r07_raygrad_hier_bench.json (or --out).
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


def fern_leg(a) -> dict:
    import cfnerf_b200 as cf
    dev = torch.device("cuda:0")
    cfg = O.CfnConfig(K=64)
    pc, pf = O.make_params(cfg, 0, "default"), O.make_params(cfg, 1, "default")
    sa, sr = O.make_latents(cfg, 0)
    H, W, focal, Nc, Nf = 756, 1008, 815.1, 64, 128
    res = {"gpu": gpu_info(), "config": "fern 8x512 F=4 K=64, two networks, NDC, 64 + 128 samples", "reps": a.reps,
           "warmup": a.warmup, "train_step_ms": {}}
    c2w = torch.eye(4)[:3].clone()
    c2w[2, 3] = 0.3
    o, d = O.get_rays(H, W, focal, c2w)
    vd = (d / d.norm(dim=-1, keepdim=True)).reshape(-1, 3)
    o, d = O.ndc_rays(H, W, focal, 1.0, o, d)
    n = H * W
    image = torch.cat([o.reshape(-1, 3), d.reshape(-1, 3), torch.zeros(n, 1), torch.ones(n, 1), vd], -1).float()
    g = torch.Generator().manual_seed(0)
    for B in (1024, 4096):
        rays = image[torch.randperm(n, generator=g)[:B]].to(dev)
        target = torch.rand(B, 3, generator=g).to(dev)
        t_rand, u = torch.rand(B, Nc, generator=g).to(dev), torch.rand(B, Nf, generator=g).to(dev)
        for prec in ("bf16", "tf32"):
            net_c = cf.NeRFFlowsParams.from_oracle_params(cfg, pc, sa, sr).to(dev)
            net_f = cf.NeRFFlowsParams.from_oracle_params(cfg, pf, sa, sr).to(dev)
            for rg in (False, True):
                def step():
                    net_c.zero_grad(set_to_none=True)
                    net_f.zero_grad(set_to_none=True)
                    r = rays.detach().requires_grad_(rg)
                    out = cf.render_rays(r, net_c, None, Nc, True, False, perturb=1., t_rand=t_rand, u=u, N_importance=Nf,
                                         network_fine=net_f, precision=prec, detach_z_samples=True)
                    coarse = dict(rgb_map=out["rgb0"], depth_map=out["depth0"], loss_entropy=out["loss_entropy0"])
                    (cf.trainer_loss(out, target, cfg.K)["loss"] + cf.trainer_loss(coarse, target, cfg.K)["loss"]).backward()
                ms = median_ms(step, a.warmup, a.reps)
                res["train_step_ms"][f"B{B}_{prec}_raygrad{int(rg)}"] = ms
                print(f"fern train step B={B} {prec} ray-grad={rg}: {ms:.3f} ms", flush=True)
            del net_c, net_f
            torch.cuda.empty_cache()
    net_c = cf.NeRFFlowsParams.from_oracle_params(cfg, pc, sa, sr).to(dev).requires_grad_(False)
    net_f = cf.NeRFFlowsParams.from_oracle_params(cfg, pf, sa, sr).to(dev).requires_grad_(False)
    pose0 = c2w.to(dev)
    idx = torch.randperm(n, generator=g)[:4096].to(dev)
    target = torch.rand(4096, 3, device=dev)

    def pose_step():
        pose = pose0.clone().requires_grad_(True)
        rays = cf.rays_from_pose(H, W, focal, pose, 0., 1., True)[idx]
        out = cf.render_rays(rays, net_c, None, Nc, False, False, N_importance=Nf, network_fine=net_f, precision="tf32",
                             detach_z_samples=True)
        ((out["rgb_map"].mean(-1) - target) ** 2).mean().backward()
    ms = median_ms(pose_step, a.warmup, a.reps)
    res["pose_step_ms"] = {"image": f"{W}x{H}", "rays": 4096, "chain": "tf32", "frozen_networks": True, "ms": ms}
    print(f"fern localisation step (4096 of {W}x{H} pixels, tf32, frozen networks): {ms:.3f} ms", flush=True)
    res["peak_memory_gb"] = torch.cuda.max_memory_allocated(dev) / 1e9
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default="africa", choices=["africa", "fern"])
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.config == "fern":
        res = fern_leg(a)
        out = a.out or os.path.join(ROOT, "profiles", "r07_raygrad_hier_bench.json")
        os.makedirs(os.path.dirname(out), exist_ok=True)
        with open(out, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res))
        return
    a.out = a.out or os.path.join(ROOT, "profiles", "r06_raygrad_bench.json")
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
