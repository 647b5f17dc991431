#!/usr/bin/env python
"""bench.py — rays/s of CF-NeRF's K-sample uncertainty render (and of its training step) on N B200s, one process per GPU.

    python bench.py --gpus N --steps K --warmup W                    # this repo's CUDA path (default config: africa)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's own code on the host CPU
    python bench.py --config fern|lego ...                           # BASELINE.json configs[3] / configs[4]
    python bench.py ... --dump-outputs DIR                           # + the last timed step's maps as DIR/*.npy
                                                                     # (rank 0's rays only when N > 1)

Configs (BASELINE.json `configs`; SURVEY §8(d)):
  africa  configs[1]: 512x512 image, N=128 samples, K=32, one image per GPU per step (weak scaling, no collective), plus
          the other half of the metric, configs[2]: one optimisation step on 4096 rays per GPU (weak), on a 4096-ray
          GLOBAL batch (strong: 4096/N rays per GPU = the reference's own N_rand = 512 at N = 8) and on 512 rays.
  fern    configs[3]: 1008x756 forward-facing image, NDC rays, 64 coarse + 128 fine samples, K=64, two networks; the rows
          of ONE image shard over the GPUs (strong scaling).
  lego    configs[4]: 800x800 views on the pose_spherical circle (200 views), K=128, white background; views go round
          robin over the GPUs, a step renders one view per GPU (weak scaling).

`value` times the device-resident path (rays in HBM -> K-field maps + mean/std/depth in HBM); `e2e` times the public
host-in / host-out call `render_rays_host` (pinned host rays in, the K fields + statistics back in pinned host memory; the
device-to-host copies of a chunk overlap the kernels of the next one).  `roofline` is the dominant
kernel (the tcgen05 network stage K1) against the measured dense bf16 peak, timed with CUDA events inside the timed
region; `roofline.kernels` adds the streaming kernels (raw2outputs, sample_pdf, flows+compositing forward / backward)
measured in the same run.  `cpu_baseline` is the UNMODIFIED reference (oracle/_ref, staged by oracle/build_ref.py) on a
bounded ray sample on this box's host cores — the oracle port when the staged copy is absent.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# The render precision of the driver's bench line: the tensor-core mode that passes EVERY parity fixture at the 2e-3 bar,
# including the SURVEY 8(d) "stressed heads" weights (tests/test_gpu_parity.py::test_bench_dtype_meets_the_bar_...).
# bf16 operands run at the same rate but drift to ~1e-2 there: the trunk's 8-bit significand, not the heads, is what
# limits it (scripts/experiments/k1_precision_sim.py).
RENDER_PRECISION = "fp16"
N_VIEWS_LEGO = 200
DUMP_BYTES = 64_000_000          # --dump-outputs: all files together stay below this

CONFIGS = {
    "africa": dict(H=512, W=512, focal=443.4, near=1.2, far=8.0, ndc=False, Nc=128, Nf=0, K=32, white_bkgd=False,
                   scaling="weak",
                   workload="africa.txt full-image 512x512 uncertainty render (mean/variance/depth), N=128 samples, K=32 "
                            "latent samples, W=512 D=8, random-init weights, one image per GPU per step"),
    "fern": dict(H=756, W=1008, focal=815.1, near=0.0, far=1.0, ndc=True, Nc=64, Nf=128, K=64, white_bkgd=False,
                 scaling="strong",
                 workload="LLFF fern-shape 1008x756 forward-facing render, NDC rays, 64 coarse + 128 fine samples (two "
                          "networks), K=64 latent samples, W=512 D=8, random-init weights, rows of ONE image sharded "
                          "over the GPUs"),
    "lego": dict(H=800, W=800, focal=1111.1, near=2.0, far=6.0, ndc=False, Nc=128, Nf=0, K=128, white_bkgd=True,
                 scaling="weak",
                 workload="Blender-lego-shape 800x800 360-degree sweep (pose_spherical, 200 views), N=128 samples, K=128 "
                          "latent samples, white background, W=512 D=8, random-init weights, views round-robin over the "
                          "GPUs, one view per GPU per step"),
}


def flop_per_point(cfg) -> int:
    """SURVEY §8(d): dense MACs of one network evaluation (amortisation once per point) x 2; 4 708 864 for the canonical net."""
    W, ip, idr, F = cfg.W, cfg.in_pos, cfg.in_dir, cfg.F
    mac = ip * W + (cfg.D - 2) * W * W + (W + (ip if cfg.skip >= 0 else 0)) * W          # trunk
    mac += W * W + W * cfg.h_alpha + (W + idr) * (W // 2) + (W // 2) * cfg.h_rgb          # feature, h_alpha, views, h_rgb
    mac += cfg.h_alpha * 4 * F + cfg.h_rgb * 18 * F                                      # amortisation (alpha 4F, rgb 18F)
    return 2 * mac


def pose_spherical(theta_deg: float, phi_deg: float, radius: float) -> torch.Tensor:
    """load_blender.py:29-34 (trans_t, rot_phi, rot_theta and the axis flip), restated for the synthetic 360-degree poses."""
    th, phi = math.radians(theta_deg), math.radians(phi_deg)
    trans = torch.eye(4)
    trans[2, 3] = radius
    rphi = torch.tensor([[1, 0, 0, 0], [0, math.cos(phi), -math.sin(phi), 0], [0, math.sin(phi), math.cos(phi), 0],
                         [0, 0, 0, 1.0]])
    rth = torch.tensor([[math.cos(th), 0, -math.sin(th), 0], [0, 1, 0, 0], [math.sin(th), 0, math.cos(th), 0],
                        [0, 0, 0, 1.0]])
    return (torch.tensor([[-1.0, 0, 0, 0], [0, 0, 1, 0], [0, 1, 0, 0], [0, 0, 0, 1]]) @ rth @ rphi @ trans)[:3]


def view_pose(config: str, index: int) -> torch.Tensor:
    if config == "lego":
        thetas = torch.linspace(-180.0, 180.0, N_VIEWS_LEGO + 1)[:-1]
        return pose_spherical(float(thetas[index % N_VIEWS_LEGO]), -30.0, 4.0)
    c2w = torch.eye(4)[:3].clone()
    if config == "fern":
        c2w[2, 3] = 0.3          # camera slightly in front of the NDC near plane origin
    if index:
        th = torch.tensor(0.05 * index)
        c2w[0, 0], c2w[0, 2], c2w[2, 0], c2w[2, 2] = torch.cos(th), torch.sin(th), -torch.sin(th), torch.cos(th)
    return c2w


def image_rays_host(config: str, index: int) -> torch.Tensor:
    """The (H*W,11) ray batch `render(H, W, focal, c2w=pose, use_viewdirs=True)` assembles (main:129-158), built on the
    host with the oracle's restatement of get_rays / ndc_rays."""
    from oracle import cfnerf_oracle as O
    c = CONFIGS[config]
    o, d = O.get_rays(c["H"], c["W"], c["focal"], view_pose(config, index))
    if not c["ndc"]:
        return O.pack_ray_batch(o, d, c["near"], c["far"])
    vd = (d / d.norm(dim=-1, keepdim=True)).reshape(-1, 3)
    o, d = O.ndc_rays(c["H"], c["W"], c["focal"], 1.0, o, d)
    n = o.reshape(-1, 3).shape[0]
    return torch.cat([o.reshape(-1, 3), d.reshape(-1, 3), torch.full((n, 1), c["near"]), torch.full((n, 1), c["far"]), vd],
                     -1).float().contiguous()


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                f = [x.strip() for x in out.split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def ncu_dram_traffic(summary_csv: str, block: int = 0):
    """dram__bytes_read.sum + dram__bytes_write.sum of kernel block `block` of a committed `ncu --set full` summary under
    profiles/ (the recipe's per-launch figure); None when the file is absent."""
    path = os.path.join(ROOT, "profiles", summary_csv)
    if not os.path.isfile(path):
        return None
    mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot, blocks = 0.0, -1
    for line in open(path):
        if line.startswith("##"):
            blocks += 1
            continue
        f = line.strip().split(",")
        if max(blocks, 0) == block and len(f) == 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            tot += float(f[2]) * mult.get(f[1], 1.0)
    return tot or None


def dump_outputs(out_dir: str, chunks, limit: int = DUMP_BYTES, seed: int = 0) -> tuple[int, int]:
    """Write what one render step returned (the dicts of its render_rays calls, concatenated along the ray axis) as
    <out_dir>/<key>.npy in float32.  When the arrays together would exceed `limit` bytes, every array keeps the same
    rows: a fixed, seeded, sorted sample of the rays, so that two builds run with the same arguments write the same
    rays.  Returns (rays written, rays rendered)."""
    import numpy as np
    keys = sorted(chunks[0])
    B = sum(c[keys[0]].shape[0] for c in chunks)
    per_ray = sum(4 * math.prod(chunks[0][k].shape[1:]) for k in keys)
    n = min(B, (limit - 4096) // per_ray)          # 4096: room for the .npy headers
    rows = None if n == B else torch.randperm(B, generator=torch.Generator().manual_seed(seed))[:n].sort().values
    os.makedirs(out_dir, exist_ok=True)
    for k in keys:
        a = torch.cat([c[k] for c in chunks], 0)
        assert a.is_floating_point(), (k, a.dtype)
        if rows is not None:
            a = a[rows.to(a.device)]
        np.save(os.path.join(out_dir, k + ".npy"), a.float().cpu().numpy())
    return n, B


def host_threads() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------------------------------------------
# the host CPU arm: the unmodified reference (oracle/_ref) when staged, else the oracle port
# ------------------------------------------------------------------------------------------------------------------
class CpuReference:
    """Times the reference's own path on the host cores.  kind "reference": `run_nerf_uncertainty_NF.render()` ->
    `batchify_rays` -> `render_rays` -> `run_network` -> `NeRF_Flows.forward` -> `raw2outputs` of the UNMODIFIED files
    staged under oracle/_ref (or /root/reference in the build container); kind "port": oracle/cfnerf_oracle.py with the
    reference's K-fold conditioning.  The coarse+fine configs have no counterpart in the reference (SURVEY A9/A10) and
    always run the port."""

    def __init__(self, config: str):
        from oracle import cfnerf_oracle as O
        from oracle import refload
        self.O, self.config, self.c = O, config, CONFIGS[config]
        torch.set_num_threads(host_threads())       # torchrun exports OMP_NUM_THREADS=1: the reference gets every core
        self.cores = torch.get_num_threads()
        self.cfg = O.CfnConfig(K=self.c["K"])
        self.p = O.make_params(self.cfg, 0, "default")
        self.sa, self.sr = O.make_latents(self.cfg, 0)
        self.p_fine = O.make_params(self.cfg, 1, "default") if self.c["Nf"] else None
        self.kind = "port"
        self.main = self.model = self.nq = None
        if not self.c["Nf"] and refload.reference_available():
            try:
                self.main, self.model, self.nq = refload.build_reference_model(self.cfg, self.p, self.sa, self.sr)
                self.kind = "reference"
            except Exception as e:      # e.g. a third-party module of the host script missing on this box
                sys.stderr.write(f"bench: unmodified reference not loadable ({e!r}); timing the oracle port\n")

    def sample_rays(self, n_rays: int) -> torch.Tensor:
        rays = image_rays_host(self.config, 0)
        return rays[:: max(1, rays.shape[0] // n_rays)][:n_rays].contiguous()

    def render(self, rays: torch.Tensor):
        O, c, cfg = self.O, self.c, self.cfg
        ea, er = O.test_latents(self.sa, self.sr)
        with torch.no_grad():
            if self.kind == "reference":
                kw = dict(is_train=False, uniformsample=False, network_query_fn=self.nq, perturb=False, N_importance=0,
                          N_samples=128, K_samples=cfg.K, network_fn=self.model, use_viewdirs=True,
                          white_bkgd=c["white_bkgd"], raw_noise_std=0., ndc=False, lindisp=False, retraw=True)  # main:382-405
                batch = torch.stack([rays[:, 0:3], rays[:, 3:6]], 0)
                rgb, disp, depth, _ = self.main.render(c["H"], c["W"], c["focal"], chunk=8192, rays=batch, near=c["near"],
                                                       far=c["far"], **kw)
                n = cfg.K
                return torch.mean(rgb, -1), torch.std(rgb, -1) * n / (n - 1), torch.mean(depth, -1)   # main:1122-1131
            outs = []
            for i in range(0, rays.shape[0], 512):          # netchunk = 65536 points (main:604)
                if c["Nf"]:
                    o = O.render_rays_hier(self.p, self.p_fine, cfg, rays[i:i + 512], ea, er, False, c["Nc"], c["Nf"],
                                           white_bkgd=c["white_bkgd"], faithful=True)
                else:
                    o = O.render_rays(self.p, cfg, rays[i:i + 512], ea, er, False, white_bkgd=c["white_bkgd"], faithful=True)
                outs.append(O.k_reduce(o["rgb_map"], o["depth_map"], cfg.K))
            return outs

    def rays_per_s(self, n_rays: int, reps: int, warm: int = 0):
        rays = self.sample_rays(n_rays)
        times = []
        for it in range(warm + reps):
            t0 = time.perf_counter()
            self.render(rays)
            if it >= warm:
                times.append(time.perf_counter() - t0)
        return rays.shape[0], times

    def train_step_seconds(self, n_rays: int, anomaly: bool):
        """One iteration of the trainer body (main:1014-1067) at the reference's own batch size on the host: render in
        train mode, K-mean + KDE-NLL + 0.01 * entropy, backward, Adam — autograd anomaly mode as shipped (ON, set at import
        by model/models.py:5) or off."""
        O, cfg = self.O, self.cfg
        rays = O.synthetic_rays(n_rays, 1)
        target = torch.rand(n_rays, 3, generator=torch.Generator().manual_seed(2))
        torch.autograd.set_detect_anomaly(bool(anomaly))
        try:
            if self.kind == "reference":
                params = list(self.model.parameters())
                opt = torch.optim.Adam(params=params, lr=5e-4, betas=(0.9, 0.999))                       # main:339
                kw = dict(is_train=True, uniformsample=False, network_query_fn=self.nq, perturb=1.0, N_importance=0,
                          N_samples=128, K_samples=cfg.K, network_fn=self.model, use_viewdirs=True, white_bkgd=False,
                          raw_noise_std=1.0, ndc=False, lindisp=False)
                batch = torch.stack([rays[:, 0:3], rays[:, 3:6]], 0)
                t0 = time.perf_counter()
                rgbs, disp, depth, extras = self.main.render(8, 8, 10.0, chunk=1024 * 32, rays=batch, near=1.2, far=8.0,
                                                             verbose=False, retraw=False, **kw)
                loss = O.kde_nll_loss(rgbs, target, extras["loss_entropy"].mean(), cfg.K, 0.01)["loss"]
                opt.zero_grad()
                loss.backward()
                opt.step()
                return time.perf_counter() - t0
            p = {k: v.clone().requires_grad_(True) for k, v in self.p.items()}
            opt = torch.optim.Adam(list(p.values()), lr=5e-4, betas=(0.9, 0.999))
            g = torch.Generator().manual_seed(3)
            t0 = time.perf_counter()
            out = O.render_rays(p, cfg, rays, torch.randn(cfg.K, 1, generator=g), torch.randn(cfg.K, 3, generator=g), True,
                                t_rand=torch.rand(n_rays, 128, generator=g), faithful=True)
            loss = O.kde_nll_loss(out["rgb_map"], target, out["loss_entropy"], cfg.K, 0.01)["loss"]
            opt.zero_grad()
            loss.backward()
            opt.step()
            return time.perf_counter() - t0
        finally:
            torch.autograd.set_detect_anomaly(False)

    def describe(self, n_rays: int) -> str:
        what = ("the UNMODIFIED reference (run_nerf_uncertainty_NF.render -> render_rays -> NeRF_Flows -> raw2outputs, staged "
                "under oracle/_ref)" if self.kind == "reference" else
                "oracle port of the reference (faithful K-fold conditioning)")
        return f"{n_rays} evenly spaced rays of the {self.c['W']}x{self.c['H']} image, {what}, torch CPU fp32, no_grad"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ref = CpuReference(args.config)
    n, times = ref.rays_per_s(args.cpu_rays, args.steps, args.warmup)
    tot = sum(times)
    v = n * len(times) / tot
    c = CONFIGS[args.config]
    line = {
        "impl": "reference", "metric": "rays/sec (K-sample uncertainty render)", "value": v, "unit": "rays/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times),
        "higher_is_better": True, "scaling": c["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": c["workload"], "rays_per_image": c["H"] * c["W"],
                   "reference_sample": f"each step times {n} evenly spaced rays of the image on the host CPU"},
        "cpu_baseline": {"value": v, "unit": "rays/s", "cores": ref.cores, "kind": ref.kind,
                         "sample": ref.describe(n) + " per step"},
        "e2e": {"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# the GPU arm
# ------------------------------------------------------------------------------------------------------------------
class K1Timer:
    """CUDA events around every network-stage launch (Engine.network) inside a timed region, on the launching stream."""

    def __init__(self):
        from cfnerf_b200.engine import Engine
        self.on, self.events, self.points = False, [], 0
        orig = Engine.network
        timer = self

        def timed(eng, B, N, *a, **k):
            if not timer.on:
                return orig(eng, B, N, *a, **k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = orig(eng, B, N, *a, **k)
            e1.record()
            timer.events.append((e0, e1))
            timer.points += B * N
            return r

        Engine.network = timed

    def total_ms(self):
        return sum(a.elapsed_time(b) for a, b in self.events)


def cuda_time_ms(fn, iters=10, warm=3):
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


def streaming_kernel_rooflines(cf, dev, net, K, N, peaks):
    """raw2outputs (K2'), sample_pdf (K3), flows + compositing forward (K2) and its backward (K4) measured in this run;
    algorithmic bytes per ray are the SURVEY §8(d) figures; inputs are larger than the 126 MB L2."""
    from cfnerf_b200.engine import _ptr, _stream
    hbm = peaks["hbm_gbs"]
    out = []
    f32 = dict(dtype=torch.float32, device=dev)
    lib = cf._lib.load()
    B = 16384
    raw = torch.randn(B, N, K, 4, device=dev)
    z = (1.2 + torch.cumsum(torch.rand(B, N, device=dev) * 0.05 + 0.01, -1)).contiguous()
    d = torch.randn(B, 3, device=dev)
    rgb, disp, depth = torch.empty(B, 3, K, **f32), torch.empty(B, K, **f32), torch.empty(B, K, **f32)
    ms = cuda_time_ms(lambda: cf._lib.check(lib.cfn_raw2outputs_f32(_ptr(raw), _ptr(z), _ptr(d), 3, 0, _ptr(rgb), _ptr(disp),
                                                                   None, _ptr(depth), B, N, K, _stream())))
    bpr = 16 * N * K + 4 * N + 12 + 20 * K
    out.append({"kernel": "raw2outputs_kernel (K2')", "bound": "hbm", "achieved": B * bpr / ms / 1e6, "peak": hbm, "unit": "GB/s",
                "frac": B * bpr / ms / 1e6 / hbm, "ms": ms, "rays": B, "bytes_per_ray": bpr})
    del raw
    B3, M, Nf = 1 << 20, 63, 128
    bins = torch.sort(torch.rand(B3, M, device=dev) * 5 + 1, -1).values
    ww, u, smp = torch.rand(B3, M - 1, device=dev), torch.rand(B3, Nf, device=dev), torch.empty(B3, Nf, **f32)
    ms = cuda_time_ms(lambda: cf._lib.check(lib.cfn_sample_pdf_f32(_ptr(bins), _ptr(ww), _ptr(u), _ptr(smp), None, B3, M, Nf,
                                                                  _stream())))
    bpr = 4 * (M + (M - 1) + Nf) + 4 * Nf
    out.append({"kernel": "sample_pdf_kernel (K3)", "bound": "hbm", "achieved": B3 * bpr / ms / 1e6, "peak": hbm, "unit": "GB/s",
                "frac": B3 * bpr / ms / 1e6 / hbm, "ms": ms, "rays": B3, "bytes_per_ray": bpr,
                "note": "latency-bound on the sequential fp32 CDF scan the bit-exactness spec fixes (124 dependent adds per ray)"})
    del bins, ww, u, smp
    eng = cf.engine_for(net, dev, RENDER_PRECISION)
    B2 = 16384
    from oracle import cfnerf_oracle as O
    rays = O.synthetic_rays(B2, 1).to(dev)
    zz = eng.zvals(rays, cf.reference_t_schedule(N, dev), None, False)
    fp = eng.network(B2, N, rays=rays, z_vals=zz)
    ea, er = cf.test_latents(net, dev)
    ms = cuda_time_ms(lambda: eng.flow_composite(fp, zz, rays[:, 3:6], 11, ea, er, False, want_kstats=True))
    bpr = 72 * 4 * N + 4 * N + 44 + 20 * K + 32
    # transcendental work per (point, k): 16 tanh + 3 sigmoid + softplus + exp, ~2 MUFU operations each in the one-MUFU
    # flavour -> ~41 MUFU ops; 16 MUFU lanes per SM per clock
    mufu_peak = 148 * 16 * (peaks.get("sm_max_mhz", 1965.0) * 1e6) / (41.0 * N * K)
    out.append({"kernel": "flow_composite_fwd_kernel (K2)", "bound": "mufu", "achieved": B2 / ms * 1e3, "peak": mufu_peak,
                "unit": "rays/s", "frac": B2 / ms * 1e3 / mufu_peak, "ms": ms, "rays": B2,
                "hbm_gbs": B2 * bpr / ms / 1e6, "hbm_frac": B2 * bpr / ms / 1e6 / hbm, "bytes_per_ray": bpr,
                "note": "transcendental-bound: ~41 MUFU operations per (point, k) at 16 lanes/clk/SM and the max SM clock"})
    o = eng.flow_composite(fp, zz, rays[:, 3:6], 11, ea, er, False, train=True, want_trans=True)
    g_rgb = torch.randn(B2, 3, K, device=dev) * 1e-3
    g_ld = torch.full((B2, 2), -0.01 / (B2 * N * K), device=dev)
    ms_f = cuda_time_ms(lambda: eng.flow_composite(fp, zz, rays[:, 3:6], 11, ea, er, False, train=True, want_trans=True))
    ms_b = cuda_time_ms(lambda: eng.flow_composite_bwd(fp, zz, rays[:, 3:6], 11, ea, er, False, g_rgb, None, g_ld, trans=o["trans"], seg_sums=o["seg_sums"]))
    bpr_b = 2 * 72 * 4 * N + 4 * N * K + 4 * N + 44 + 12 * K + 32      # records in, record gradients out, transmittances in
    out.append({"kernel": "flow_composite_fwd_kernel<train> (K2, with log-dets + transmittance output)", "bound": "mufu",
                "achieved": B2 / ms_f * 1e3, "unit": "rays/s", "ms": ms_f, "rays": B2})
    out.append({"kernel": "flow_composite_bwd_kernel (K4)", "bound": "issue", "achieved": B2 / ms_b * 1e3, "unit": "rays/s",
                "ms": ms_b, "rays": B2, "ratio_to_forward": ms_b / ms_f, "hbm_gbs": B2 * bpr_b / ms_b / 1e6,
                "hbm_frac": B2 * bpr_b / ms_b / 1e6 / hbm, "bytes_per_ray": bpr_b,
                "note": "recompute + adjoint + 18F-row lane reduction per point: instruction-issue bound, not HBM-bound"})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="africa", choices=sorted(CONFIGS))
    ap.add_argument("--precision", default=RENDER_PRECISION, choices=["bf16", "fp16", "tf32", "fp32"],
                    help="operand type of the tensor-core GEMM chain (bf16 and fp16 run at the same rate)")
    ap.add_argument("--chunk", type=int, default=0, help="rays per render_rays call (0: sized so that the flow-parameter "
                                                         "buffer of one call holds ~4.2 M points)")
    ap.add_argument("--cpu-rays", type=int, default=2048)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training legs (BASELINE.json configs[2])")
    ap.add_argument("--no-kernels", action="store_true", help="skip the per-kernel streaming rooflines")
    ap.add_argument("--train-rays", type=int, default=4096, help="rays per GPU per optimisation step (weak-scaling leg)")
    ap.add_argument("--train-rays-global", type=int, default=4096,
                    help="global batch of the strong-scaling training leg (BASELINE configs[2]: 4096 rays over all GPUs)")
    ap.add_argument("--train-precision", default="bf16", choices=["bf16", "tf32", "fp32"],
                    help="GEMM engine of the training legs: bf16 storage + kind::f16 (BASELINE configs[2] wording), "
                         "tf32 over fp32 storage, or the fp32 CUDA-core check engine")
    ap.add_argument("--no-graph", action="store_true", help="launch the training step eagerly instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed render steps, write the maps the last one returned as DIR/<name>.npy (float32; "
                         f"rank 0; a fixed seeded sample of the rays when all of them exceed {DUMP_BYTES / 1e6:.0f} MB)")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the outputs of the CUDA path; it has no meaning with --impl reference")
        return run_reference(args)

    import torch.distributed as dist

    import cfnerf_b200 as cf
    from oracle import cfnerf_oracle as O

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (no CPU fallback); use --impl reference for the host baseline")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    c = CONFIGS[args.config]
    cfg = O.CfnConfig(K=c["K"])
    Nc, Nf, K = c["Nc"], c["Nf"], c["K"]
    n_eval = Nc + (Nc + Nf if Nf else 0)                 # network evaluations per ray (coarse grid + merged fine grid)
    FPP = flop_per_point(cfg)
    sa, sr = O.make_latents(cfg, 0)
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, O.make_params(cfg, 0, "default"), sa, sr).to(dev)   # random init
    net_fine = cf.NeRFFlowsParams.from_oracle_params(cfg, O.make_params(cfg, 1, "default"), sa, sr).to(dev) if Nf else None
    timer = K1Timer()
    chunk = args.chunk or max(1024, (4194304 // max(n_eval - Nc, Nc)) // 1024 * 1024)

    # ---- this rank's rays per step -------------------------------------------------------------------------------
    H, W = c["H"], c["W"]
    if args.config == "fern":        # strong scaling: contiguous row blocks of ONE image
        from cfnerf_b200 import dist as D
        lo, hi = D.shard_bounds(H, rank, world)
        full = image_rays_host("fern", 0)
        views_host = [full[lo * W:hi * W].contiguous().pin_memory()]
        rays_total_per_step = H * W
    elif args.config == "lego":      # weak scaling: a different view per GPU per step, round robin over the 200 poses
        n_views = min(args.steps + max(args.warmup, 3), 4)    # distinct poses actually generated (host memory)
        views_host = [image_rays_host("lego", (s * world + rank)).pin_memory() for s in range(n_views)]
        rays_total_per_step = H * W * world
    else:
        views_host = [image_rays_host("africa", rank).pin_memory()]
        rays_total_per_step = H * W * world
    views_dev = [v.to(dev) for v in views_host]
    B = views_dev[0].shape[0]
    render_kw = dict(K_samples=K, white_bkgd=c["white_bkgd"], precision=args.precision, want_kstats=True)
    if Nf:
        render_kw.update(N_importance=Nf, network_fine=net_fine)

    def render_device(rays):
        """device-resident step through the public API: per chunk z schedule -> K1 -> K2 (-> K3 -> K1 -> K2)."""
        return [cf.render_rays(rays[i:i + chunk], net, None, Nc, False, False, **render_kw) for i in range(0, rays.shape[0], chunk)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    launches_per_chunk = 3 if not Nf else 9      # zvals, K1, K2 [+ mean_over_k, sample_pdf, merge, K1, K2 and the t-grid]
    n_chunks = (B + chunk - 1) // chunk
    W_ = max(args.warmup, 3)
    for s in range(W_):
        render_device(views_dev[s % len(views_dev)])
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    timer.on = True
    ev0.record()
    outs = None
    for s in range(args.steps):
        del outs            # the previous step's maps go back to the allocator first, as in the warm-up loop
        outs = render_device(views_dev[(W_ + s) % len(views_dev)])
    ev1.record()
    barrier()
    timer.on = False
    ms = ev0.elapsed_time(ev1)
    k1_ms, k1_points, n_k1 = timer.total_ms(), timer.points, len(timer.events)
    if args.dump_outputs and rank == 0 and outs:
        n, n_all = dump_outputs(args.dump_outputs, outs)
        sys.stderr.write(f"bench: wrote the maps of {n} of the {n_all} rays of the last timed step to {args.dump_outputs}\n")
    del outs

    # ---- end to end through the public API: pinned host rays in, K fields + statistics out ----
    out_host = None
    keys = ("rgb_map", "disp_map", "depth_map", "kstats")

    def render_e2e(rays_host):
        # the public host-in / host-out call: H2D of a chunk, render_rays, D2H of its outputs on a second stream (the
        # copies of chunk i overlap the kernels of chunk i + 1); returns once the last byte is in pinned host memory
        nonlocal out_host
        out_host = cf.render_rays_host(rays_host, net, Nc, chunk=chunk, keys=keys, out=out_host, **render_kw)
        torch.cuda.synchronize()
        return out_host

    for s in range(2):
        render_e2e(views_host[s % len(views_host)])
    barrier()
    ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ee0.record()
    for s in range(args.steps):
        cat = render_e2e(views_host[(2 + s) % len(views_host)])
    ee1.record()
    barrier()
    e2e_ms = ee0.elapsed_time(ee1)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    h2d = views_host[0].numel() * 4
    d2h = sum(v.numel() * 4 for v in cat.values())
    del cat, out_host
    torch.cuda.empty_cache()

    # ---- the other half of the metric: optimisation steps (BASELINE.json configs[2]); africa only ----
    # render (train mode, saved activations) -> K-mean + KDE-NLL + 0.01 * entropy -> backward (flow/composite backward,
    # dgrad chain, split-K wgrad) -> one all-reduce of the flat gradient bucket (N > 1) -> Adam -> weight re-pack, replayed
    # from CUDA graphs.  Runs last (it moves the weights).
    train = {}
    do_train = args.config == "africa" and not args.no_train
    if do_train:
        from cfnerf_b200 import dist as D
        legs = [("train_step", args.train_rays, "weak", f"{args.train_rays} rays per GPU"),
                ("train_step_strong", max(1, args.train_rays_global // world), "strong",
                 f"{args.train_rays_global}-ray global batch, {max(1, args.train_rays_global // world)} rays per GPU "
                 "(BASELINE configs[2]; = the reference's N_rand = 512 at 8 GPUs)"),
                ("train_step_512", 512, "weak", "512 rays per GPU: the reference's own batch size (train_NF.sh:6)")]
        seen = {}
        for name, n_t, scaling, what in legs:
            if n_t in seen:                      # e.g. N = 1: the strong leg is the weak leg
                train[name] = dict(train[seen[n_t]], scaling=scaling, what=what, same_run_as=seen[n_t])
                continue
            seen[n_t] = name
            net_t = cf.NeRFFlowsParams.from_oracle_params(cfg, O.make_params(cfg, 0, "default"), sa, sr).to(dev)
            trainer = D.FusedTrainStep(net_t, lr=5e-4, precision=args.train_precision, use_graph=not args.no_graph)
            gt = torch.Generator().manual_seed(100 + rank)
            t_rays = views_dev[0][torch.randperm(B, generator=gt)[:n_t].to(dev)].contiguous()
            t_target = torch.rand(t_rays.shape[0], 3, generator=gt).to(dev)
            torch.manual_seed(100 + rank)   # every rank draws its own latent noise, like every DataParallel replica
            for _ in range(4):
                trainer.step(t_rays, t_target, want_loss=False)
            barrier()
            te0, te1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            te0.record()
            for _ in range(args.steps):
                trainer.step(t_rays, t_target, want_loss=False)
            te1.record()
            barrier()
            t_out = trainer.step(t_rays, t_target)
            # every rank must hold bit-identical weights after the same all-reduced updates
            chk = trainer.weights_checksum()
            same = True
            if world > 1:
                allc = [torch.empty_like(chk) for _ in range(world)]
                dist.all_gather(allc, chk)
                same = all(torch.equal(allc[0], x) for x in allc)
                if not same:
                    raise SystemExit(f"bench: ranks hold different weights after the {name} leg: {[x.tolist() for x in allc]}")
            tm = torch.tensor([te0.elapsed_time(te1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            step_s = float(tm) * 1e-3 / args.steps
            train[name] = {"value": n_t * world / step_s, "unit": "rays/s", "ms_per_step": step_s * 1e3, "rays_per_gpu": n_t,
                           "global_batch_rays": n_t * world, "scaling": scaling, "what": what,
                           "precision": args.train_precision, "cuda_graph": not args.no_graph, "loss": float(t_out["loss"]),
                           "achieved_tflops_per_gpu": n_t * 128 * FPP * 3 / step_s / 1e12,
                           "ranks_hold_identical_weights": bool(same), "weights_checksum": [float(x) for x in chk]}
            del trainer, net_t
            torch.cuda.empty_cache()

    # one trunk-layer forward GEMM of the training step timed alone (burst peak applies: 10 back-to-back launches)
    tg = None
    if do_train and args.train_precision in ("tf32", "bf16") and rank == 0:
        Mp = args.train_rays * 128
        bf = args.train_precision == "bf16"
        dt = torch.bfloat16 if bf else torch.float32
        Xg = torch.randn(Mp, cfg.W, device=dev).to(dt)
        Wg = (torch.randn(cfg.W, cfg.W, device=dev) * 0.05).to(dt)
        bg = torch.randn(cfg.W, device=dev)
        Yg = torch.empty(Mp, cfg.W, device=dev, dtype=dt)
        mb = torch.zeros(Mp, (cfg.W + 31) // 32, dtype=torch.int32, device=dev)
        if bf:
            tg_ms = cuda_time_ms(lambda: cf.gemm_bf16(Xg, Wg.t(), bias=bg, epilogue="relu", mask_out=mb, out=Yg))
        else:
            tg_ms = cuda_time_ms(lambda: cf.gemm(Xg, Wg.t(), engine="tf32", bias=bg, epilogue="relu", out=Yg, round_out=True))
        tg = (tg_ms, Mp, bf)
        del Xg, Yg, mb
    kernels = []
    if rank == 0 and not args.no_kernels:
        kernels = streaming_kernel_rooflines(cf, dev, net, K, 128, measured_peaks()[0])
    barrier()

    t = torch.tensor([ms, e2e_ms, k1_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms, k1_ms = [float(x) for x in t.cpu()]

    if rank == 0:
        peaks, which = measured_peaks()
        rays_total = rays_total_per_step * args.steps
        value = rays_total / (ms * 1e-3)
        e2e = rays_total / (e2e_ms * 1e-3)
        k1_avg_s = (k1_ms * 1e-3) / max(n_k1, 1)
        pts_per_launch = k1_points / max(n_k1, 1)
        achieved = pts_per_launch * FPP / k1_avg_s / 1e12
        peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
        line = {
            "metric": "rays/sec (K-sample uncertainty render)", "value": value, "unit": "rays/s", "n_gpus": world,
            "steps": args.steps, "warmup": W_, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": c["scaling"], "vs_baseline": None, "dtype": args.precision,
            "data": "synthetic",
            "config": {"workload": c["workload"], "name": args.config, "rays_per_step_per_gpu": B,
                       "rays_per_step_total": rays_total_per_step, "chunk_rays": chunk, "network_evaluations_per_ray": n_eval,
                       "l2": f"no flush needed: each step streams a {B * (n_eval - Nc if Nf else Nc) * 288 / 1e9:.1f} GB "
                             "flow-parameter buffer (>> 126 MB L2)"},
            "e2e": {"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches_per_chunk * n_chunks * args.steps,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak,
                         "traffic": ncu_dram_traffic("r02_prof_k1_summary.csv") if (args.config == "africa" and not args.chunk) else None,
                         "traffic_note": "DRAM bytes of one K1 launch (4 194 304 points) from profiles/r02_prof_k1_summary.csv "
                                         "(ncu --set full of this command); algorithmic HBM bytes = 288 B/point of flow "
                                         "parameters written = 1.208e9",
                         "kernel": "mlp_tc_kernel (network stage K1)",
                         "flop_per_point": FPP, "points_per_launch": pts_per_launch, "launches_timed": n_k1,
                         "avg_launch_ms": k1_avg_s * 1e3,
                         "peak_source": f"{which}: bf16_tflops_sustained (K1 is timed inside a long step)",
                         "frac_of_burst_peak": achieved / peaks.get("bf16_tflops", peak),
                         "k1_share_of_step": k1_ms / ms, "whole_step_tflops": value / world * n_eval * FPP / 1e12,
                         "kernels": kernels},
            "clocks": sampler.summary(),
        }
        if do_train:
            line["train_step"] = train["train_step"]
            line["train_step"]["note"] = (
                "forward + loss + backward + all-reduce + Adam + re-pack through cfnerf_b200.dist.FusedTrainStep; GEMMs = "
                "TMA-fed tcgen05: kind::f16 over bf16-stored activations / gradients (bf16), kind::tf32 over fp32 storage "
                "(tf32), or CUDA-core fp32 FMA (fp32); fp32 accumulation, master weights and weight gradients throughout; "
                "flops = 3 x forward")
            line["train_step_strong"] = train["train_step_strong"]
            line["train_step_512"] = train["train_step_512"]
            if tg is not None:
                tg_ms, Mp, bf = tg
                esz = 2 if bf else 4
                gb = 2.0 * Mp * cfg.W * esz / 1e9          # activations in + out (the weight matrix is L2-resident)
                tf = 2.0 * Mp * cfg.W * cfg.W / (tg_ms * 1e-3) / 1e12
                hbm = peaks.get("hbm_gbs", 6545.9)
                tpeak = peaks.get("bf16_tflops", peaks.get("bf16_tflops_sustained"))     # burst: the GEMM is timed alone
                roof = ({"bound": "tensor", "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": tf / tpeak,
                         "peak_source": f"{which}: bf16_tflops (burst; this GEMM is timed alone)",
                         "hbm_gbs": gb / (tg_ms * 1e-3), "hbm_frac": gb / (tg_ms * 1e-3) / hbm} if bf else
                        {"bound": "hbm", "achieved": gb / (tg_ms * 1e-3), "peak": hbm, "unit": "GB/s",
                         "frac": gb / (tg_ms * 1e-3) / hbm, "tflops": tf})
                roof.update({
                    "traffic": ncu_dram_traffic("r01_prof_tgemm_fwd_summary.csv" if not bf else "r01_prof_tgemm_bf16_summary.csv")
                    if Mp == 524288 else None,
                    "traffic_note": "DRAM read + write of this GEMM from the committed ncu --set full capture "
                                    "(profiles/r01_prof_tgemm_*_summary.csv) at 524288 points; algorithmic bytes = "
                                    f"2 x points x 512 x {esz} = {2 * 524288 * 512 * esz:.4g}",
                    "kernel": "tgemm_kernel (one trunk-layer forward GEMM of the training step: bias + ReLU + bit mask)",
                    "ms": tg_ms})
                line["train_step"]["roofline"] = roof
        if not args.no_cpu_baseline and world == 1:
            ref = CpuReference(args.config)
            n, times = ref.rays_per_s(args.cpu_rays if not Nf else min(args.cpu_rays, 256), 2)
            line["cpu_baseline"] = {"value": n / min(times), "unit": "rays/s", "cores": ref.cores, "kind": ref.kind,
                                    "sample": ref.describe(n) + ", best of 2"}
            if do_train:
                on, off = ref.train_step_seconds(512, True), ref.train_step_seconds(512, False)
                line["cpu_baseline_train"] = {
                    "value": 512 / on, "unit": "rays/s", "cores": ref.cores, "kind": ref.kind,
                    "anomaly_mode_on_rays_per_s": 512 / on, "anomaly_mode_off_rays_per_s": 512 / off,
                    "sample": "one 512-ray iteration of the trainer body (render in train mode, KDE-NLL + 0.01 * entropy, "
                              "backward, Adam; main:1014-1067) on the host; autograd anomaly mode ON as shipped "
                              "(model/models.py:5) = `value`, and OFF"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
