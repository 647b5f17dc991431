"""What a field-space query (cfnerf_b200.query_field / field_grid, F6) costs on one GPU.

On the africa architecture (8x512, F = 4) with `default`-variant weights, fp16 (the render default), at K = 32 and
K = 128:
  grid        field_grid over a 256^3 grid (16.8 M points, the default chunk of 4 194 304 points): wall time of the
              whole call ending in a device synchronise, alternated reps times -> points/s end to end
  kernels     CUDA events around K1 (cfn_network_fwd, explicit points) and the stats kernel (cfn_field_stats_f32) on one
              chunk of 4 194 304 points (1.2 GB of flow records: larger than the 126 MB L2), iters launches each
  k2          K2 (cfn_flow_composite_fwd, render flavour with kstats) on 32 768 rays x 128 samples at the same K, for
              its time per (sample, k) next to the stats kernel's time per (point, k)
  baseline    run_network (raw (M,K,4) in HBM) + the reduction over k in torch on one chunk of 2 097 152 points,
              against query_field on the same points (and the largest difference between the two)

Writes profiles/r04_field_bench.json (or --out) with the card's name, power limit and max SM clock.
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

PRECISION = "fp16"
GRID = 256
CHUNK = 1 << 22
BASELINE_POINTS = 1 << 21
BOUNDS = ((-1.5, 1.5), (-1.5, 1.5), (-1.5, 1.5))


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()
    return {"query": q[0], "value": q[1] if len(q) > 1 else ""}


def timed(fn) -> float:
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def event_ms(fn, iters: int) -> float:
    fn()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1) / iters


def case(cf, K: int, dev, reps: int, iters: int) -> dict:
    cfg = O.CfnConfig(K=K)
    p = O.make_params(cfg, 0, "default")
    sa, sr = O.make_latents(cfg, 0)
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev)
    eng = cf.engine_for(net, dev, PRECISION)
    eps_a, eps_c = cf.test_latents(net, dev)
    out = {"K": K, "precision": PRECISION, "grid": GRID, "chunk": CHUNK}

    # ---- end to end: field_grid over 256^3 ----
    def grid():
        r = cf.field_grid(net, BOUNDS, GRID, precision=PRECISION)
        del r

    grid()                                                     # warm-up: module load, weight packing
    t = [timed(grid) for _ in range(reps)]
    out["grid_s"] = t
    out["grid_points_per_s"] = GRID ** 3 / statistics.median(t)

    # ---- K1 vs the stats kernel on one chunk ----
    g = torch.Generator(device=dev).manual_seed(K)
    pts = (torch.rand(CHUNK, 3, device=dev, generator=g) * 3 - 1.5).contiguous()
    vd = torch.nn.functional.normalize(torch.randn(CHUNK, 3, device=dev, generator=g), dim=-1).contiguous()
    fp = eng.network(CHUNK, 1, pts=pts, viewdirs=vd)
    stats = torch.empty(CHUNK, 8, device=dev)
    k1_ms = event_ms(lambda: eng.network(CHUNK, 1, pts=pts, viewdirs=vd), iters)
    st_ms = event_ms(lambda: eng.field_stats(fp, eps_a, eps_c, out=stats), iters)
    out["chunk_k1_ms"] = k1_ms
    out["chunk_stats_ms"] = st_ms
    out["k1_points_per_s"] = CHUNK / (k1_ms * 1e-3)
    out["stats_ns_per_point_k"] = st_ms * 1e6 / (CHUNK * K)
    out["stats_share_of_k1_plus_stats"] = st_ms / (k1_ms + st_ms)
    del fp

    # ---- K2 at the same K: time per (sample, k) ----
    B, N = 32768, 128
    rays = O.synthetic_rays(B, 5).to(dev)
    z = eng.zvals(rays, cf.reference_t_schedule(N, dev), None, False)
    fpr = eng.network(B, N, rays=rays, z_vals=z)
    k2_ms = event_ms(lambda: eng.flow_composite(fpr, z, rays[:, 3:6], 11, eps_a, eps_c, False, want_kstats=True), iters)
    out["k2_rays"], out["k2_samples_per_ray"] = B, N
    out["k2_ms"] = k2_ms
    out["k2_ns_per_sample_k"] = k2_ms * 1e6 / (B * N * K)
    del fpr, z, rays

    # ---- baseline: raw samples to HBM, then the reduction in torch ----
    n = BASELINE_POINTS
    bp, bv = pts[:n].contiguous(), vd[:n].contiguous()

    def baseline():
        raw, _ = cf.run_network(bp[:, None, :], bv, net, False, True, precision=PRECISION)
        x = torch.cat([torch.nn.functional.softplus(raw[:, 0, :, 3:4]), torch.sigmoid(raw[:, 0, :, 0:3])], -1)  # (n,K,4)
        m, s = x.mean(1), (x.std(1) if K > 1 else torch.zeros_like(x[:, 0]))
        return torch.stack([m[:, 0], s[:, 0], m[:, 1], m[:, 2], m[:, 3], s[:, 1], s[:, 2], s[:, 3]], -1)

    def mine():
        return cf.query_field(bp, net, bv, precision=PRECISION)["stats"]

    ref, got = baseline(), mine()
    out["baseline_max_abs_diff"] = (ref - got).abs().max().item()
    del ref, got
    torch.cuda.reset_peak_memory_stats(dev)
    base0 = torch.cuda.memory_allocated(dev)
    tb = [timed(baseline) for _ in range(reps)]
    out["baseline_peak_extra_bytes"] = torch.cuda.max_memory_allocated(dev) - base0
    torch.cuda.reset_peak_memory_stats(dev)
    tq = [timed(mine) for _ in range(reps)]
    out["query_field_peak_extra_bytes"] = torch.cuda.max_memory_allocated(dev) - base0
    out["baseline_points"] = n
    out["baseline_raw_bytes"] = n * K * 16
    out["baseline_s"], out["query_field_s"] = tb, tq
    out["baseline_points_per_s"] = n / statistics.median(tb)
    out["query_field_points_per_s"] = n / statistics.median(tq)
    del net, eng, pts, vd, stats
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_field_bench.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("field_bench.py measures on a CUDA device; none is visible")
    import cfnerf_b200 as cf
    dev = torch.device("cuda:0")
    result = {"gpu": gpu_info(), "architecture": "africa (D=8, W=512, F=4, h_alpha=h_rgb=64), default-variant weights",
              "cases": []}
    for K in (32, 128):
        result["cases"].append(case(cf, K, dev, args.reps, args.iters))
        print(json.dumps(result["cases"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
