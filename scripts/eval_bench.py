"""What the F5 evaluation (cfnerf_b200.evaluate) costs next to the render it evaluates, on one GPU.

For the lego-like view (800x800, K = 128, white background) and the africa view (512x512, K = 32) of bench.py, with the
canonical network (random init) in bench.py's render precision and seeded uniform targets (the cost does not depend on
the values):
  render     the chunked render with want_kstats (what a user runs anyway to look at a view)
  evaluate   evaluate_view on the same rays: render + trainer-loss pass + records + one sparsification call + host syncs
The two are alternated, three times each; the difference of the medians is the evaluation's cost.  Then
cfn_sparsification_f32 alone (CUDA events, preallocated workspace) at V = 1 and V = 8 views of 640 000 pixels, and, for
context, the host route a user had before: render_rays_host of the K fields, then the numpy fp64 restatement of the
metrics (tests/eval_oracle.py) in chunks of 65 536 pixels.

Writes profiles/r03_eval_bench.json (or the path given with --out) with the card's name, power limit and max SM clock.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench                                   # noqa: E402
import eval_oracle as E                        # noqa: E402
from oracle import cfnerf_oracle as O          # noqa: E402

CHUNK = 32768


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


def view_case(cf, config: str, dev, reps: int, host_route: bool) -> dict:
    c = bench.CONFIGS[config]
    cfg = O.CfnConfig(K=c["K"])
    p = O.make_params(cfg, 0, "default")
    sa, sr = O.make_latents(cfg, 0)
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev)
    rays_host = bench.image_rays_host(config, 0)
    P = rays_host.shape[0]
    rays = rays_host.to(dev)
    target = torch.rand(P, 3, generator=torch.Generator().manual_seed(1)).to(dev)
    kw = dict(N_samples=c["Nc"], white_bkgd=c["white_bkgd"], precision=bench.RENDER_PRECISION)

    def render():
        for i in range(0, P, CHUNK):
            o = cf.render_rays(rays[i:i + CHUNK], net, want_kstats=True, **kw)
            del o

    res = {}

    def evaluate():
        res.update(cf.evaluate_view(rays, target, net, chunk=CHUNK, **kw))

    render(), evaluate()                                       # warm-up: module load, weight packing, CUB tuning
    t_r, t_e = [], []
    for _ in range(reps):
        t_r.append(timed(render))
        t_e.append(timed(evaluate))
    out = {"pixels": P, "K": c["K"], "N_samples": c["Nc"], "precision": bench.RENDER_PRECISION, "chunk": CHUNK,
           "render_kstats_s": t_r, "evaluate_view_s": t_e,
           "median_render_s": statistics.median(t_r), "median_evaluate_s": statistics.median(t_e),
           "evaluation_cost_s": statistics.median(t_e) - statistics.median(t_r),
           "metrics": {k: res[k] for k in ("psnr", "nll", "ause_rmse", "ause_mae")}}
    if host_route:
        t0 = time.perf_counter()
        h = cf.render_rays_host(rays_host, net, chunk=CHUNK, keys=("rgb_map",), **kw)
        t1 = time.perf_counter()
        recs, tgt = [], target.cpu().numpy()
        for i in range(0, P, 65536):
            recs.append(E.eval_records(h["rgb_map"][i:i + 65536].numpy(), None, tgt[i:i + 65536], None, c["K"]))
        rec = {k: np.concatenate([r[k] for r in recs]) for k in ("uncertainty", "sq_err", "abs_err", "nll_map")}
        sp = E.sparsification(rec["uncertainty"], rec["sq_err"], rec["abs_err"], 100)
        t2 = time.perf_counter()
        out["host_route"] = {"render_rays_host_s": t1 - t0, "numpy_metrics_s": t2 - t1, "total_s": t2 - t0,
                             "bytes_to_host": int(P * 3 * c["K"] * 4),
                             "ause_rmse": sp["ause_rmse"], "ause_mae": sp["ause_mae"]}
    del net
    torch.cuda.empty_cache()
    return out


def sparsify_alone(dev, V: int, P: int, iters: int) -> dict:
    from cfnerf_b200 import _lib
    from cfnerf_b200.engine import _ptr
    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(V)
    u, e, a = (torch.rand(V, P, device=dev, generator=g) for _ in range(3))
    need = C.c_size_t()
    _lib.check(lib.cfn_sparsification_workspace_bytes(V, P, 100, C.byref(need)))
    ws = torch.empty(need.value, dtype=torch.uint8, device=dev)
    curves, ause = torch.empty(V, 4, 100, device=dev), torch.empty(V, 2, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call():
        _lib.check(lib.cfn_sparsification_f32(_ptr(u), _ptr(e), _ptr(a), V, P, 100, _ptr(ws), ws.numel(), _ptr(curves),
                                              _ptr(ause), stream))

    for _ in range(3):
        call()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        call()
    t1.record()
    t1.synchronize()
    return {"V": V, "P": P, "S": 100, "workspace_bytes": need.value, "ms_per_call": t0.elapsed_time(t1) / iters,
            "input_bytes": V * P * 12,
            "note": "inputs + workspace fit the 126 MB L2" if V * P * 12 + need.value < 126e6 else "working set larger than L2"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_eval_bench.json"))
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_bench.py measures on a CUDA device; none is visible")
    import cfnerf_b200 as cf
    dev = torch.device("cuda:0")
    torch.set_num_threads(bench.host_threads())
    result = {"gpu": gpu_info(), "views": {}, "sparsification_alone": []}
    for config in ("lego", "africa"):
        result["views"][config] = view_case(cf, config, dev, args.reps, host_route=True)
        print(config, json.dumps(result["views"][config]), flush=True)
    for V in (1, 8):
        result["sparsification_alone"].append(sparsify_alone(dev, V, 640000, 50))
        print(json.dumps(result["sparsification_alone"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
