"""Drop-in surface: the reference's own callables, same names / argument meaning / return contract, backed by
the CUDA library through the C-ABI (include/cfnerf_b200.h).

    render_rays   run_nerf_uncertainty_NF.py:457-553
    run_network   run_nerf_uncertainty_NF.py:67-85
    raw2outputs   run_nerf_uncertainty_NF.py:411-454
    sample_pdf    extension (the reference kept only the comment run_nerf_helpers.py:9-11; upstream nerf-pytorch
                  semantics, specified by oracle/cfnerf_oracle.py::sample_pdf)
    install(mod)  rebinds `mod.render_rays` / `mod.raw2outputs` so the unmodified `render()` / `train()` use them.

Extra keyword-only arguments (never required by the reference's callers) expose what the reference draws
implicitly, so tests can inject it: `t_rand`, `eps_alpha`, `eps_rgb`, `u`, and `precision`.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib
from ._lib import check
from .engine import Engine, _f32c, _ptr, _stream, _unwrap, engine_for

# fp16 operands have an 11-bit significand (TF32-class) at the same tensor-core rate as bf16: with trained-like
# ("stressed") conditioning heads bf16 drifts to 1e-2 on the predictive mean while fp16 stays at 1e-3, inside the
# 2e-3 bar (tests/test_gpu_parity.py::test_stressed_heads_precision_report).  "bf16" and "fp32" remain selectable.
DEFAULT_PRECISION = "fp16"
# Training (forward with saved activations + backward) runs layer by layer: "fp32" = CUDA-core FMA GEMMs (the exact
# check mode), "tf32" / "bf16" / "fp16" = tcgen05 kind::tf32 GEMMs over fp32 storage with tf32-rounded operands.
DEFAULT_TRAIN_PRECISION = "tf32"
# points per network call of the reference: netchunk_per_gpu (65536, main:604) x n_gpus (main:336); it decides how many
# independent latent draws a training batch sees (see render_rays)
DEFAULT_NETCHUNK = 1024 * 64


# ------------------------------------------------------------------------------------------------------
# schedules and latents (host-side plumbing, mirrors the reference lines cited)
# ------------------------------------------------------------------------------------------------------
def reference_t_schedule(n_samples: int, device) -> torch.Tensor:
    """main:510 — the hard-coded 96+32 schedule (the reference requires N_samples == 128, main:516).  For any other
    N_samples (extension, SURVEY A10) the upstream linspace(0,1,N) schedule is used.  Computed on the CPU in fp32 like
    the oracle, then moved: torch's CUDA linspace may differ in the last bit."""
    key = (int(n_samples), str(device))
    t = _T_SCHEDULES.get(key)
    if t is None:       # cached per device: a pageable host-to-device copy per call would stall the host every step
        if n_samples == 128:
            t = torch.cat([torch.linspace(0., 0.5, steps=97)[:-1], torch.linspace(0.5, 1., steps=32)], 0)
        else:
            t = torch.linspace(0., 1., steps=n_samples)
        t = _T_SCHEDULES[key] = t.to(device)
    return t


_T_SCHEDULES: dict = {}


def test_latents(module, device):
    """models.py:198-205 — constructor-time draws with the LAST sample's noise forced to zero."""
    ea = module.sample_alpha.detach().clone().float()
    er = module.sample_rgb.detach().clone().float()
    ea[-1] = 0
    er[-1] = 0
    return ea.reshape(-1).to(device).contiguous(), er.to(device).contiguous()


# ------------------------------------------------------------------------------------------------------
# stand-alone kernels
# ------------------------------------------------------------------------------------------------------
def raw2outputs(raw, z_vals, rays_d, raw_noise_std=0, white_bkgd=False, pytest=False):
    """main:411-454.  raw (B,N,K,4), z_vals (B,N), rays_d (B,3) -> rgb_map (B,3,K), disp_map (B,K),
    weights (B,N,K), depth_map (B,K).  `raw_noise_std` only consumes RNG in the reference (the noise is never
    added, main:432-442); it is accepted and ignored."""
    lib = _lib.load()
    if not raw.is_cuda:
        raise RuntimeError("cfnerf_b200.raw2outputs needs CUDA tensors (no CPU fallback)")
    dev = raw.device
    raw, z_vals, rays_d = _f32c(raw, dev), _f32c(z_vals, dev), _f32c(rays_d, dev)
    B, N, K, four = raw.shape
    assert four == 4 and z_vals.shape == (B, N) and rays_d.shape == (B, 3)
    f32 = dict(dtype=torch.float32, device=dev)
    rgb, disp = torch.empty(B, 3, K, **f32), torch.empty(B, K, **f32)
    w, depth = torch.empty(B, N, K, **f32), torch.empty(B, K, **f32)
    with torch.cuda.device(dev):
        check(lib.cfn_raw2outputs_f32(_ptr(raw), _ptr(z_vals), _ptr(rays_d), 3, int(bool(white_bkgd)), _ptr(rgb),
                                      _ptr(disp), _ptr(w), _ptr(depth), B, N, K, _stream()), "cfn_raw2outputs_f32")
    return rgb, disp, w, depth


def sample_pdf(bins, weights, N_samples, det=False, pytest=False, *, u=None, return_below=False):
    """Upstream signature `sample_pdf(bins, weights, N_samples, det, pytest)`.  bins (B,M), weights (B,M-1) ->
    samples (B,N_samples); `u` (B,N_samples) overrides the uniforms (det -> linspace(0,1,N), else torch.rand)."""
    lib = _lib.load()
    dev = bins.device
    if dev.type != "cuda":
        raise RuntimeError("cfnerf_b200.sample_pdf needs CUDA tensors (no CPU fallback)")
    bins, weights = _f32c(bins, dev), _f32c(weights, dev)
    B, M = bins.shape
    assert weights.shape == (B, M - 1)
    if u is None:
        if det:
            u = torch.linspace(0., 1., steps=N_samples).to(dev).expand(B, N_samples)
        else:
            u = torch.rand(B, N_samples, device=dev)
    u = _f32c(u, dev)
    out = torch.empty(B, N_samples, dtype=torch.float32, device=dev)
    below = torch.empty(B, N_samples, dtype=torch.int32, device=dev) if return_below else None
    with torch.cuda.device(dev):
        check(lib.cfn_sample_pdf_f32(_ptr(bins), _ptr(weights), _ptr(u), _ptr(out), _ptr(below), B, M, N_samples,
                                     _stream()), "cfn_sample_pdf_f32")
    return (out, below) if return_below else out


def merge_sorted(z_a, z_b, *, return_src=False):
    """sort(cat[z_a, z_b], -1) per ray.  return_src: also the permutation src (B,Na+Nb) int32, the index into
    cat[z_a, z_b] of every output slot (torch.sort(stable=True).indices) -> (out, src)."""
    lib = _lib.load()
    dev = z_a.device
    z_a, z_b = _f32c(z_a, dev), _f32c(z_b, dev)
    B, Na = z_a.shape
    Nb = z_b.shape[1]
    out = torch.empty(B, Na + Nb, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        if return_src:
            src = torch.empty(B, Na + Nb, dtype=torch.int32, device=dev)
            check(lib.cfn_merge_sorted_src_f32(_ptr(z_a), _ptr(z_b), _ptr(out), _ptr(src), B, Na, Nb, _stream()),
                  "cfn_merge_sorted_src_f32")
            return out, src
        check(lib.cfn_merge_sorted_f32(_ptr(z_a), _ptr(z_b), _ptr(out), B, Na, Nb, _stream()), "cfn_merge_sorted_f32")
    return out


def mean_over_k(w):
    lib = _lib.load()
    dev = w.device
    w = _f32c(w, dev)
    rows, K = w.numel() // w.shape[-1], w.shape[-1]
    out = torch.empty(w.shape[:-1], dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        check(lib.cfn_mean_over_k_f32(_ptr(w), _ptr(out), rows, K, _stream()), "cfn_mean_over_k_f32")
    return out


# ------------------------------------------------------------------------------------------------------
# training: one autograd node around network + flows + compositing
# ------------------------------------------------------------------------------------------------------
class _RenderTrainFn(torch.autograd.Function):
    """forward: cfn_network_fwd(save) + cfn_flow_composite_fwd(train); backward: cfn_flow_composite_bwd +
    cfn_network_bwd.  The parameters are inputs so that autograd writes into the reference module's own .grad.
    eps_a (G,K) / eps_c (G,K,3): one latent draw per group of `group_rays` rays (0: G = 1).
    sched = (t_vals, t_rand or None, lindisp, merged): what made z_vals from the rays.  merged is None for a grid
    cfn_zvals_f32 made, or (src, Nc) for the fine pass's merged grid (src from merge_sorted(..., return_src=True), kept
    alive here for the backward; t_vals / t_rand are then the coarse pass's).  When the rays need a gradient the
    backward runs the ray flavour instead (cfn_flow_composite_bwd_rays + cfn_network_bwd_inputs + cfn_ray_grad_f32 or
    cfn_ray_grad_merged_f32), without any weight gradient when no parameter needs one."""

    @staticmethod
    def forward(ctx, eng: Engine, rays, z_vals, eps_a, eps_c, white_bkgd, want_weights, group_rays, sched, *params):
        B, N = z_vals.shape
        fp, ws = eng.network(B, N, rays=rays, z_vals=z_vals, save=True)
        out = eng.flow_composite(fp, z_vals, rays[:, 3:6], 11, eps_a, eps_c, white_bkgd, want_raw=True,
                                 want_weights=want_weights, train=True, eps_group_rays=group_rays, want_trans=True)
        ctx.eng, ctx.white_bkgd, ctx.group_rays, ctx.sched = eng, white_bkgd, group_rays, sched
        sg = out["seg_sums"] if out["seg_sums"] is not None else torch.empty(0, device=rays.device)
        ctx.save_for_backward(rays, z_vals, eps_a, eps_c, fp, ws, out["trans"], sg)
        w = out["weights"] if want_weights else torch.empty(0, device=rays.device)
        ctx.mark_non_differentiable(out["disp_map"], out["raw"], w)
        # logdet_sums (B,2): per-ray sums of the alpha / rgb log-det terms (the entropy scalars are built from them)
        return out["rgb_map"], out["disp_map"], out["depth_map"], out["raw"], out["logdet_sums"], w

    @staticmethod
    def backward(ctx, g_rgb, g_disp, g_depth, g_raw, g_ld, g_w):
        eng = ctx.eng
        rays, z_vals, eps_a, eps_c, fp, ws, trans, sg = ctx.saved_tensors
        B, N = z_vals.shape
        dev = rays.device
        g_rgb = _f32c(g_rgb, dev) if g_rgb is not None else torch.zeros(B, 3, eng.K, device=dev)
        g_depth = _f32c(g_depth, dev) if g_depth is not None else None
        # the per-ray log-det gradient seeds stay on the device: reading them back would stall the host once per step
        gl = _f32c(g_ld.detach(), dev) if g_ld is not None else torch.zeros(B, 2, device=dev)
        g_rays = None
        with torch.cuda.device(dev):
            if not ctx.needs_input_grad[1]:
                g_fp, g_glob = eng.flow_composite_bwd(fp, z_vals, rays[:, 3:6], 11, eps_a, eps_c, ctx.white_bkgd, g_rgb,
                                                      g_depth, gl, trans=trans, eps_group_rays=ctx.group_rays,
                                                      seg_sums=sg if sg.numel() else None)
                grads = eng.network_bwd(g_fp, B, N, ws)
            else:
                g_fp, g_glob, g_zd, g_dl = eng.flow_composite_bwd(
                    fp, z_vals, rays[:, 3:6], 11, eps_a, eps_c, ctx.white_bkgd, g_rgb, g_depth, gl, trans=trans,
                    eps_group_rays=ctx.group_rays, seg_sums=sg if sg.numel() else None, ray_terms=True)
                need_w = any(ctx.needs_input_grad[9:])
                grads, g_enc = eng.network_bwd_inputs(g_fp, B, N, ws, weights=need_w)
                t_vals, t_rand, lindisp, merged = ctx.sched
                g_rays = eng.ray_grad(rays, z_vals, t_vals, t_rand, lindisp, g_enc, g_zd, g_dl, merged=merged)
                if not need_w:
                    return (None, g_rays) + (None,) * (7 + len(eng.params))
        gg = g_glob.sum(0)
        grads[0], grads[1] = gg[0:1], gg[1:2]
        grads[2], grads[3] = gg[2:5], gg[5:8]
        grads = [g.reshape(p.shape) for g, p in zip(grads, eng.params)]
        return (None, g_rays, None, None, None, None, None, None, None, *grads)


def latent_groups(B: int, N: int, netchunk: int):
    """How the reference's `batchify` (main:47-64) cuts a training batch of B rays x N samples into network calls of
    `netchunk` points, each of which draws its own latent noise (models.py:233-251): -> (rays per call, number of
    calls).  Whole rays per call need N | netchunk — true for the reference's only N (128 | 65536); otherwise (the
    192-sample fine grid of the extension) the batch is treated as one call."""
    if netchunk and netchunk % N == 0 and B * N > netchunk:
        r = netchunk // N
        return r, (B + r - 1) // r
    return 0, 1


# Latent draws per ray up to which the fused network + compositing kernel is faster than K1 -> K2 (see
# fused_composite): its two compositing warps per CTA have two tile-times per tile of rays, which covers K = 32 (one
# latent group per ray) with room to spare but not K = 128, where they would set the pace of the kernel.
FUSED_MAX_K = 32


def fused_composite(eng, N: int, need_weights: bool, group_rays: int) -> bool:
    """Test-mode render passes that run network + compositing as one kernel (Engine.network(..., composite=)):
    tensor-core precision, no weights / raw output, whole rays per 128-point tile, the compiled F = 4 flavour, one
    latent-draw set for every ray and K <= FUSED_MAX_K.  Everything else keeps the two launches."""
    return (eng.precision in ("fp16", "bf16") and not need_weights and 128 % N == 0 and eng.F == 4 and group_rays == 0
            and eng.K <= FUSED_MAX_K)


def _latent_draws(module, K: int, device, train: bool, G: int, eps_alpha, eps_rgb, batch: str):
    """The base latent draws of a batch that makes G network calls -> (eps_a, eps_c): (K), (K,3) when G = 1, else
    (G,K), (G,K,3).  Without eps_alpha: in train mode one fresh (alpha, rgb) pair per network call, drawn in the
    reference's order (models.py:234, 246); in test mode the constructor-time draws.  The caller's eps_alpha / eps_rgb
    may be (K,1) / (K,3) (one call) or (G,K,1) / (G,K,3) (one pair per call).  `batch` describes the batch in errors."""
    if eps_alpha is None:
        if train:
            pairs = [(torch.empty([K, 1], device=device).normal_(),                            # models.py:234
                      torch.empty([K, 3], device=device).normal_()) for _ in range(G)]        # models.py:246
            eps_alpha, eps_rgb = torch.stack([a for a, _ in pairs], 0), torch.stack([c for _, c in pairs], 0)
        else:
            eps_alpha, eps_rgb = test_latents(module, device)
    if eps_rgb.dim() == 3:      # (G,K,3): the caller fixed the draws of every network call
        if eps_rgb.shape[0] != G:
            raise ValueError(f"{eps_rgb.shape[0]} latent draws given but the batch makes {G} network calls ({batch})")
        eps_a, eps_c = _f32c(eps_alpha.reshape(G, -1), device), _f32c(eps_rgb, device)
        return (eps_a[0].contiguous(), eps_c[0].contiguous()) if G == 1 else (eps_a, eps_c)
    if G > 1:
        raise ValueError(f"the batch makes {G} network calls: pass eps_alpha (G,K,1) and eps_rgb (G,K,3)")
    return _f32c(eps_alpha.reshape(-1), device), _f32c(eps_rgb.reshape(-1, 3), device)


def _entropy_base_terms(module, eps_a, eps_c):
    """base log-densities of models.py:268/283 (no 2*pi term), written like the reference so autograd gives the same
    gradient for the global std parameters.  eps_a (K) / eps_c (K,3) -> two scalars; with a leading group axis
    ((G,K) / (G,K,3)) -> two (G,) tensors, one pair per network call."""
    a_mean, a_std = module.alpha_mean, module.alpha_std
    c_mean, c_std = module.rgb_mean, module.rgb_std
    grouped = eps_c.dim() == 3
    ea = eps_a.reshape(eps_c.shape[0], -1, 1) if grouped else eps_a.reshape(1, -1, 1)
    ec = eps_c if grouped else eps_c[None]
    a0 = ea * a_std + a_mean
    c0 = ec * c_std + c_mean
    base_a = -0.5 * (a_std.log() * 2 + (a0 - a_mean) * (a0 - a_mean) * (a_std ** 2).reciprocal())
    base_c = -0.5 * (c_std.log() * 2 + (c0 - c_mean) * (c0 - c_mean) * (c_std ** 2).reciprocal())
    ba, bc = base_a.mean((1, 2)), base_c.mean((1, 2))
    return (ba, bc) if grouped else (ba[0], bc[0])


def _entropy_rows(module, eps_a, eps_c, logdet_sums, B, N, K, group_rays):
    """The (B*N, K, 1) `loss_entropy` tensor `render_rays` returns in train mode: every network call's entropy scalar
    (models.py:286) broadcast over the rows of that call (models.py:291; cat in batchify, main:57-62)."""
    if not group_rays:
        base_a, base_c = _entropy_base_terms(module, eps_a.reshape(-1), eps_c.reshape(-1, 3))
        ld = logdet_sums.sum(0)
        cnt = float(B * N * K)
        ent = base_a - ld[0] / cnt + base_c - ld[1] / cnt
        return ent.expand(B * N, K, 1)
    G = eps_c.shape[0]
    base_a, base_c = _entropy_base_terms(module, eps_a, eps_c)                                 # (G,), (G,)
    sizes = torch.tensor([min(group_rays, B - g * group_rays) for g in range(G)], device=logdet_sums.device)
    gid = torch.repeat_interleave(torch.arange(G, device=logdet_sums.device), sizes)
    ld = torch.zeros(G, 2, device=logdet_sums.device, dtype=logdet_sums.dtype).index_add(0, gid, logdet_sums)
    cnt = sizes.to(ld.dtype) * float(N * K)
    ent = base_a - ld[:, 0] / cnt + base_c - ld[:, 1] / cnt                                    # (G,)
    return torch.repeat_interleave(ent, sizes * N)[:, None, None].expand(B * N, K, 1)


# ------------------------------------------------------------------------------------------------------
# run_network / render_rays
# ------------------------------------------------------------------------------------------------------
def run_network(inputs, viewdirs, fn, is_val, is_test, embed_fn=None, embeddirs_fn=None, netchunk=1024 * 64, *,
                eps_alpha=None, eps_rgb=None, precision=None):
    """main:67-85.  inputs (B,N,3), viewdirs (B,3) -> (outputs (B,N,K,4) [rgb|sigma raw], loss_entropy).
    `embed_fn` / `embeddirs_fn` are accepted for signature compatibility (the encoding is fused into the network
    kernel).  `netchunk` does not chunk anything here (memory is bounded inside the library); it only decides, in
    train mode, how many independent latent draws / entropy scalars the batch sees, as in the reference (one per
    `batchify` call of netchunk points).  Test mode returns zeros for
    loss_entropy like the reference (models.py:223); train mode returns the entropy scalar broadcast to (B*N,K,1)
    (models.py:291) — use render_rays for a differentiable training step."""
    module = _unwrap(fn)
    dev = inputs.device
    eng = engine_for(fn, dev, precision or DEFAULT_PRECISION)
    B, N = inputs.shape[0], inputs.shape[1]
    pts = _f32c(inputs.reshape(-1, 3), dev)
    if viewdirs is None:
        raise ValueError("the reference model requires use_viewdirs (model/models.py:63-64)")
    vd = _f32c(viewdirs.reshape(-1, 3), dev)
    if vd.shape[0] != B:
        raise ValueError("viewdirs must be (B,3): one direction per ray (main:74-76)")
    train = not is_test
    # train mode: one latent draw per batchify call of `netchunk` points (main:47-64, models.py:233-251)
    group_rays, G = latent_groups(B, N, int(netchunk)) if train else (0, 1)
    eps_a, eps_c = _latent_draws(module, eng.K, dev, train, G, eps_alpha, eps_rgb,
                                 f"{B} rays x {N} samples, netchunk {netchunk}")
    with torch.cuda.device(dev), torch.no_grad():
        fp = eng.network(B, N, pts=pts, viewdirs=vd)
        # raw comes out of the flow stage; compositing outputs are discarded here (z/dirs are dummies)
        z_dummy = torch.zeros(B, N, device=dev)
        out = eng.flow_composite(fp, z_dummy, vd, 3, eps_a, eps_c, False, want_raw=True, train=train,
                                 eps_group_rays=group_rays)
    raw = out["raw"]
    if not train:
        return raw, torch.zeros_like(raw)
    with torch.no_grad():
        ent = _entropy_rows(module, eps_a, eps_c, out["logdet_sums"], B, N, eng.K, group_rays)
    return raw, ent


def render_rays(ray_batch, network_fn, network_query_fn=None, N_samples=128, is_train=False, uniformsample=False,
                retraw=False, lindisp=False, K_samples=0, perturb=0., N_importance=0, network_fine=None,
                white_bkgd=False, raw_noise_std=0., verbose=False, pytest=False, *, t_rand=None, eps_alpha=None,
                eps_rgb=None, u=None, precision=None, want_weights=False, want_kstats=False, netchunk=None,
                detach_z_samples=False):
    """main:457-553, plus the coarse+fine extension when N_importance > 0 and network_fine is given (SURVEY A9/A10).

    Returns the reference dict: rgb_map (B,3,K), disp_map (B,K), depth_map (B,K); when is_train also raw
    (B,N,K,4), loss_entropy (B*N,K,1) (the per-call scalar broadcast, models.py:291) and pts (B,N,3).
    `network_query_fn` is accepted and ignored (encoding + chunking are fused).

    `netchunk` (default: the reference's netchunk_per_gpu * 1 GPU = 65536, main:336, 604; `install(..., netchunk=)`
    changes it) only matters in train mode, and only for what the reference's chunking makes observable: every
    network call of netchunk points draws its own latent noise (models.py:233-251) and returns its own entropy scalar,
    so a training batch of more than netchunk / N rays uses one (eps_alpha, eps_rgb) pair per group of netchunk / N
    rays, drawn in the reference's order, and `loss_entropy` carries one scalar per group.  `eps_alpha` / `eps_rgb` may
    be passed as (K,1) / (K,3) (one call) or (G,K,1) / (G,K,3) (one pair per call).

    A ray_batch that requires a gradient makes the maps differentiable in it (F7).  For the coarse+fine pass this needs
    detach_z_samples=True: upstream nerf-pytorch's hierarchical step, in which the resampled depths (sample_pdf of the
    detached coarse weights) are constants and the coarse depths keep their gradient through the sort.  Both passes
    then add their terms to ray_batch.grad; about 26 KB of saved activations per point on the tf32 chain, for the coarse
    and the fine points alike."""
    module = _unwrap(network_fn)
    dev = ray_batch.device
    hier = N_importance > 0 and network_fine is not None
    # F7: the rays need a gradient -> the training kernels run in test mode too (the reference's render_rays is one
    # autograd graph from ray_batch in both modes); the coarse+fine pass only with the resampled depths held constant
    ray_grad = ray_batch.requires_grad and torch.is_grad_enabled()
    if ray_grad and hier and not detach_z_samples:
        raise ValueError("ray gradients cover single-network passes by default: the coarse+fine pass (N_importance > 0 "
                         "with network_fine) is differentiable in ray_batch only with detach_z_samples=True (the "
                         "resampled depths held constant, as upstream nerf-pytorch)")
    if ray_grad and want_kstats:
        raise ValueError("want_kstats is not available together with ray gradients (ray_batch.requires_grad)")
    prec = precision or DEFAULT_PRECISION
    if is_train or ray_grad:
        prec = precision or DEFAULT_TRAIN_PRECISION
    eng = engine_for(network_fn, dev, prec)
    if K_samples and K_samples != eng.K:
        raise ValueError(f"K_samples={K_samples} but the network was built with K={eng.K}")
    rays = _f32c(ray_batch, dev)
    if rays.shape[-1] != 11:
        raise ValueError("ray_batch must be (B,11) = [o d near far viewdir] (use_viewdirs, main:504-507)")
    B = rays.shape[0]
    if B == 0 and not is_train:
        # an empty ray batch (a ragged last shard): empty maps of the right shapes, no launches
        K, f32 = eng.K, dict(dtype=torch.float32, device=dev)
        ret = {"rgb_map": torch.empty(0, 3, K, **f32), "disp_map": torch.empty(0, K, **f32), "depth_map": torch.empty(0, K, **f32)}
        if hier:
            ret.update(rgb0=torch.empty(0, 3, K, **f32), disp0=torch.empty(0, K, **f32), depth0=torch.empty(0, K, **f32),
                       z_samples=torch.empty(0, N_importance, **f32), z_vals=torch.empty(0, N_samples + N_importance, **f32))
        if want_weights:
            ret["weights"] = torch.empty(0, N_samples + (N_importance if hier else 0), K, **f32)
        if want_kstats:
            ret["kstats"] = torch.empty(0, 8, **f32)
        return ret
    with torch.cuda.device(dev):
        t_vals = reference_t_schedule(N_samples, dev)
        if perturb > 0. and t_rand is None:
            t_rand = torch.rand(B, N_samples, device=dev)                                     # main:524
            if pytest:
                import numpy as np
                t_rand = torch.Tensor(np.random.rand(B, N_samples)).to(dev)                  # main:527-530
        if t_rand is not None:
            t_rand = _f32c(t_rand, dev)
        z_vals = eng.zvals(rays, t_vals, t_rand if perturb > 0. or t_rand is not None else None, lindisp)
        sched = (t_vals, t_rand, bool(lindisp))
        # latent draws: one pair per network call of the reference (train mode), the constructor-time draws in test mode
        group_rays, G = (0, 1)
        if is_train and not hier:
            group_rays, G = latent_groups(B, N_samples, DEFAULT_NETCHUNK if netchunk is None else int(netchunk))
        eps_a, eps_c = _latent_draws(module, eng.K, dev, is_train, G, eps_alpha, eps_rgb,
                                     f"{B} rays x {N_samples} samples, netchunk {netchunk or DEFAULT_NETCHUNK}")
        if is_train and raw_noise_std > 0.:
            # the reference draws noise here and never adds it (main:432-442); same count keeps the RNG stream aligned
            torch.randn(B, N_samples, eng.K, device=dev)

        def one_pass(net, z, train, need_w, merged=None):
            e = engine_for(net, dev, prec)
            N = z.shape[1]
            if train or ray_grad:
                rgb, disp, depth, raw, ld, w = _RenderTrainFn.apply(e, rays, z, eps_a, eps_c, bool(white_bkgd),
                                                                    need_w, group_rays, sched + (merged,), *e.params)
                if not train:       # test mode with ray gradients: the maps (and weights), as the reference returns
                    return dict(rgb_map=rgb, disp_map=disp, depth_map=depth, weights=w if need_w else None)
                ent = _entropy_rows(_unwrap(net), eps_a, eps_c, ld, B, N, e.K, group_rays)    # models.py:286-291
                return dict(rgb_map=rgb, disp_map=disp, depth_map=depth, raw=raw, weights=w if need_w else None,
                            loss_entropy=ent)
            with torch.no_grad():
                if fused_composite(e, N, need_w, group_rays):
                    return e.network(B, N, rays=rays, z_vals=z, composite=dict(
                        rays_d=rays[:, 3:6], rays_d_stride=11, eps_alpha=eps_a, eps_rgb=eps_c, white_bkgd=bool(white_bkgd),
                        want_kstats=want_kstats))
                fp = e.network(B, N, rays=rays, z_vals=z)
                return e.flow_composite(fp, z, rays[:, 3:6], 11, eps_a, eps_c, bool(white_bkgd),
                                        want_raw=False, want_weights=need_w, want_kstats=want_kstats)

        if not hier:
            o = one_pass(network_fn, z_vals, is_train, want_weights)
            ret = {"rgb_map": o["rgb_map"], "disp_map": o["disp_map"], "depth_map": o["depth_map"]}
            if want_weights:
                ret["weights"] = o["weights"]
            if want_kstats and o.get("kstats") is not None:
                ret["kstats"] = o["kstats"]
            N = N_samples
        else:
            oc = one_pass(network_fn, z_vals, is_train, True)
            with torch.no_grad():
                w_mean = mean_over_k(oc["weights"])                                            # (B,Nc): shared fine grid
                z_mid = .5 * (z_vals[..., 1:] + z_vals[..., :-1])
                z_samples = sample_pdf(z_mid, w_mean[..., 1:-1], N_importance, det=(perturb == 0.), pytest=pytest,
                                       u=u)
                if ray_grad:        # the fine pass's ray gradient routes each slot back through the permutation
                    z_all, src = merge_sorted(z_vals, z_samples, return_src=True)
                else:
                    z_all = merge_sorted(z_vals, z_samples)
            o = one_pass(network_fine, z_all, is_train, want_weights, (src, N_samples) if ray_grad else None)
            ret = {"rgb_map": o["rgb_map"], "disp_map": o["disp_map"], "depth_map": o["depth_map"],
                   "rgb0": oc["rgb_map"], "disp0": oc["disp_map"], "depth0": oc["depth_map"],
                   "z_samples": z_samples, "z_vals": z_all}
            if want_weights:
                ret["weights"] = o["weights"]
            if want_kstats and o.get("kstats") is not None:
                ret["kstats"] = o["kstats"]
            if is_train:
                ret["loss_entropy0"] = oc["loss_entropy"]
            z_vals = z_all
            N = z_all.shape[1]
        if is_train:
            ret["raw"] = o["raw"]
            ret["loss_entropy"] = o["loss_entropy"]                                            # (B*N,K,1), models.py:291
            ret["pts"] = rays[:, None, 0:3] + rays[:, None, 3:6] * z_vals[..., :, None]       # main:534
    return ret


class _RaysFromPoseFn(torch.autograd.Function):
    """rays_from_pose with a gradient for c2w: backward = cfn_rays_from_pose_bwd_f32 (c2w read on the device)."""

    @staticmethod
    def forward(ctx, c2w, H, W, focal, near, far, ndc, device):
        ctx.save_for_backward(c2w)
        ctx.args = (H, W, focal, ndc, device)
        return _rays_from_pose(H, W, focal, c2w.detach(), near, far, ndc, device)

    @staticmethod
    def backward(ctx, g_rays):
        (c2w,) = ctx.saved_tensors
        H, W, focal, ndc, dev = ctx.args
        lib = _lib.load()
        c = _f32c(c2w.detach()[:3, :4], dev)
        g = torch.empty(3, 4, dtype=torch.float32, device=dev)
        partials = torch.empty(3072, dtype=torch.float32, device=dev)       # CFN_POSE_BWD_PARTIALS
        with torch.cuda.device(dev):
            check(lib.cfn_rays_from_pose_bwd_f32(int(H), int(W), float(focal), _ptr(c), int(bool(ndc)), 1.0,
                                                 _ptr(_f32c(g_rays, dev)), _ptr(partials), _ptr(g), _stream()),
                  "cfn_rays_from_pose_bwd_f32")
        gc = torch.zeros(c2w.shape, dtype=c2w.dtype, device=c2w.device)
        gc[:3, :4] = g.to(device=c2w.device, dtype=c2w.dtype)
        return gc, None, None, None, None, None, None, None


def rays_from_pose(H, W, focal, c2w, near=0., far=1., ndc=False, device=None):
    """The ray batch `render(H, W, focal, c2w=pose, use_viewdirs=True)` assembles (main:129-158) — (H*W,11) on the
    device, generated by one kernel from the 3x4 pose instead of six (H,W,3) torch intermediates.  When c2w is a tensor
    that requires a gradient (and grad mode is on) the rays carry a grad_fn whose backward is the adjoint kernel, so
    render_rays / render_image become differentiable in the pose."""
    dev = torch.device(device) if device is not None else (c2w.device if isinstance(c2w, torch.Tensor) and c2w.is_cuda
                                                           else torch.device("cuda", torch.cuda.current_device()))
    if isinstance(c2w, torch.Tensor) and c2w.requires_grad and torch.is_grad_enabled():
        return _RaysFromPoseFn.apply(c2w, H, W, focal, near, far, ndc, dev)
    return _rays_from_pose(H, W, focal, c2w, near, far, ndc, dev)


def _rays_from_pose(H, W, focal, c2w, near, far, ndc, dev):
    lib = _lib.load()
    c = torch.as_tensor(c2w, dtype=torch.float32).detach().cpu()[:3, :4].contiguous()
    rays = torch.empty(H * W, 11, dtype=torch.float32, device=dev)
    arr = (C.c_float * 12)(*c.reshape(-1).tolist())
    with torch.cuda.device(dev):
        check(lib.cfn_rays_from_pose_f32(int(H), int(W), float(focal), arr, float(near), float(far), int(bool(ndc)), 1.0,
                                         _ptr(rays), _stream()), "cfn_rays_from_pose_f32")
    return rays


def render_image(H, W, focal, c2w, network_fn, near=0., far=1., ndc=False, chunk=1024 * 32, **render_kwargs):
    """`render(H, W, focal, chunk, c2w=pose, near=, far=, use_viewdirs=True, **render_kwargs_test)` (main:103-170,
    the full-image branch): returns [rgb_map (H,W,3,K), disp_map (H,W,K), depth_map (H,W,K), extras]."""
    dev = next(_unwrap(network_fn).parameters()).device
    rays = rays_from_pose(H, W, focal, c2w, near, far, ndc, dev)
    rets = [render_rays(rays[i:i + chunk], network_fn, **render_kwargs) for i in range(0, rays.shape[0], chunk)]
    allr = {k: torch.cat([r[k] for r in rets], 0) for k in rets[0]}
    for k in allr:
        if k not in ("loss_entropy", "loss_entropy_uniformsample"):
            allr[k] = allr[k].reshape([H, W] + list(allr[k].shape[1:]))
    ex = ["rgb_map", "disp_map", "depth_map"]
    return [allr[k] for k in ex] + [{k: v for k, v in allr.items() if k not in ex}]


_COPY_STREAMS: dict = {}


def render_rays_host(rays_host, network_fn, N_samples=128, chunk=1024 * 32, keys=("rgb_map", "disp_map", "depth_map"),
                     out=None, device=None, **render_kwargs):
    """Host in, host out: what `render()` + the `.cpu()` calls of `render_path_train` do (main:129-170, 305-320), as a
    three-stage pipeline.  `rays_host` (B,11) lives in (preferably pinned) host memory; every chunk of rays is copied to
    the device, rendered by `render_rays` (test mode) and its outputs are copied back into pinned host tensors ON A
    SECOND STREAM, so that the device-to-host traffic of chunk i (20 K bytes per ray: 1.6 GB per 800 x 800 image at
    K = 128) overlaps the kernels of chunk i + 1 instead of following the last one.

    Returns {key: pinned host tensor (B, ...)} for `keys` (any of the render_rays outputs, e.g. "kstats" with
    want_kstats=True).  `out`: a dict returned by an earlier call of the same shape, to reuse its pinned buffers.
    The call returns after the last copy has completed."""
    dev = torch.device(device) if device is not None else next(_unwrap(network_fn).parameters()).device
    if dev.type != "cuda":
        raise RuntimeError("cfnerf_b200.render_rays_host needs the network on a CUDA device (no CPU fallback)")
    B = rays_host.shape[0]
    with torch.cuda.device(dev):
        main = torch.cuda.current_stream(dev)
        side = _COPY_STREAMS.get(dev)
        if side is None:
            side = _COPY_STREAMS[dev] = torch.cuda.Stream(dev)
        out = {} if out is None else out
        if B == 0:
            o = render_rays(rays_host.to(dev), network_fn, None, N_samples, False, False, **render_kwargs)
            return {k: o[k].cpu() for k in keys}
        for i in range(0, B, chunk):
            n = min(chunk, B - i)
            r = rays_host[i:i + n].to(dev, non_blocking=True)
            o = render_rays(r, network_fn, None, N_samples, False, False, **render_kwargs)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                for k in keys:
                    v = o[k]
                    if k not in out or out[k].shape[0] != B or out[k].shape[1:] != v.shape[1:]:
                        out[k] = torch.empty((B,) + tuple(v.shape[1:]), dtype=v.dtype).pin_memory()
                    out[k][i:i + n].copy_(v, non_blocking=True)
                    v.record_stream(side)       # the allocator may not hand this block out before the copy has run
        side.synchronize()
    return out


def configure(precision: str | None = None, train_precision: str | None = None, netchunk: int | None = None):
    """Module defaults used when a call does not say otherwise: render precision ("fp16" | "bf16" | "tf32" | "fp32"),
    training precision ("tf32" | "bf16" | "fp32") and the reference's netchunk (points per network call, main:336)."""
    global DEFAULT_PRECISION, DEFAULT_TRAIN_PRECISION, DEFAULT_NETCHUNK
    if netchunk is not None:        # args.netchunk_per_gpu * args.n_gpus of the host script (main:336)
        DEFAULT_NETCHUNK = int(netchunk)
    if precision is not None:
        DEFAULT_PRECISION = precision
    if train_precision is not None:
        DEFAULT_TRAIN_PRECISION = train_precision


def install(ref_module, precision: str | None = None, train_precision: str | None = None, netchunk: int | None = None):
    """Rebind the reference's module-global names (SURVEY §8(b)): `batchify_rays` looks `render_rays` up by global
    name (main:93) and `render_rays` looks `raw2outputs` up the same way (main:540).  `precision` selects the render
    mode ("fp16" default, "bf16", "tf32", "fp32"), `train_precision` the training mode ("tf32" default, "fp32")."""
    configure(precision, train_precision, netchunk)
    ref_module.render_rays = render_rays
    ref_module.raw2outputs = raw2outputs
    return ref_module


# ------------------------------------------------------------------------------------------------------
# A11: the caller's K-reduction and KDE-NLL loss (main:1027-1050), kept in torch for round 1 (SURVEY F1)
# ------------------------------------------------------------------------------------------------------
class _TrainerLossFn(torch.autograd.Function):
    """cfn_trainer_loss_f32: KDE-NLL + mse over the colour rays and the depth squared error over the depth rays in one
    kernel, both gradient seeds computed in the same pass.  depth_map may be None when there are no depth rays."""

    @staticmethod
    def forward(ctx, rgb_map, depth_map, target, target_depth):
        lib = _lib.load()
        dev = rgb_map.device
        x, t = _f32c(rgb_map.detach(), dev), _f32c(target, dev)
        d = _f32c(depth_map.detach(), dev) if depth_map is not None else None
        B, _, K = x.shape
        B_rgb = t.shape[0]
        B_depth = B - B_rgb
        td = _f32c(target_depth, dev) if B_depth else None
        if B_depth and td.shape[0] != B_depth:
            raise ValueError(f"{B} rays rendered, {B_rgb} colour targets, {td.shape[0]} depth targets")
        partial = torch.empty(B, 3, dtype=torch.float32, device=dev)
        g_rgb, g_depth = torch.empty_like(x), (torch.empty_like(d) if d is not None else None)
        with torch.cuda.device(dev):
            check(lib.cfn_trainer_loss_f32(_ptr(x), _ptr(d), _ptr(t), _ptr(td), B_rgb, B_depth, K, 1.0 / (3.0 * B_rgb),
                                           (1.0 / B_depth) if B_depth else 0.0, _ptr(partial), _ptr(g_rgb), _ptr(g_depth),
                                           _stream()), "cfn_trainer_loss_f32")
        ctx.save_for_backward(g_rgb, g_depth)
        tot = partial.sum(0)
        nll, mse = tot[0] / (3.0 * B_rgb), tot[1] / (3.0 * B_rgb)
        dl = tot[2] / B_depth if B_depth else tot[2] * 0
        ctx.mark_non_differentiable(mse)
        return nll, mse, dl

    @staticmethod
    def backward(ctx, g_nll, g_mse, g_dl):
        g_rgb, g_depth = ctx.saved_tensors
        return g_rgb * g_nll, (g_depth * g_dl if g_depth is not None else None), None, None


def trainer_loss(out, target_s, K, beta1=0.01, target_depth=None, depth_lambda=0.0):
    """The loss of the trainer body, main:1018-1055, on the dict `render_rays(cat[colour rays, depth rays], ...)`
    returned in train mode.  With depth supervision (--colmap_depth) the batch is [N_batch colour rays | depth rays]
    (main:1009-1011): colours / entropy use the first N_batch entries (main:1021-1023 — note that `extras[x][:N_batch]`
    slices the ROWS of the (B*N,K,1) entropy tensor, i.e. the first network call's scalar), the depth loss is
    `img2mse(mean_K depth_map[N_batch:], target_depth)` weighted by depth_lambda (main:1020, 1053-1054)."""
    B = out["rgb_map"].shape[0]
    B_depth = 0 if target_depth is None else int(target_depth.shape[0])
    N_batch = B - B_depth
    nll, mse, dl = _TrainerLossFn.apply(out["rgb_map"], out["depth_map"], target_s, target_depth)
    ent_rows = out["loss_entropy"]
    ent = ent_rows[:N_batch].mean() if B_depth else ent_rows.mean()
    loss = nll + beta1 * ent if beta1 else nll
    res = {"loss_nll": nll, "mse": mse, "psnr": -10. * torch.log(mse) / math.log(10.), "loss_entropy": ent}
    if B_depth:
        loss = loss + depth_lambda * dl
        res["depth_loss"] = dl
    res["loss"] = loss
    return res


def kde_nll_loss(rgb_map, target, loss_entropy, K, beta1=0.01, fused=None):
    """main:1027-1050.  On CUDA tensors the K-reduction, the KDE-NLL and its gradient run in one kernel (F1, the
    trainer loss kernel without depth rays); the torch expression below is the CPU form used by the host-side tests."""
    if fused is None:
        fused = rgb_map.is_cuda
    if fused:
        nll, mse, _ = _TrainerLossFn.apply(rgb_map, None, target, None)
        psnr = -10. * torch.log(mse) / math.log(10.)
        loss = nll + beta1 * loss_entropy.mean() if beta1 else nll
        return {"loss": loss, "loss_nll": nll, "mse": mse, "psnr": psnr}
    eps = 1e-05
    rgb_mean = rgb_map.mean(-1)
    mse = torch.mean((rgb_mean - target) ** 2)
    psnr = -10. * torch.log(mse) / math.log(10.)
    rgb_std = torch.std(rgb_map, -1) * K / (K - 1)                                            # main:1034
    h = (rgb_std.detach() * (0.8 / K) ** (-1. / 7.) + eps)[..., None]                         # main:1036
    p1 = torch.exp(-((rgb_map - target[..., None]) ** 2) / (2 * h * h))
    p2 = (2 * math.pi) ** (-1.5) / h
    nll = -torch.log((p1 * p2).mean(-1) + eps).mean()
    loss = nll + beta1 * loss_entropy.mean() if beta1 else nll
    return {"loss": loss, "loss_nll": nll, "mse": mse, "psnr": psnr}


# ---------------------------------------------------------------------------------------------------------
# the dense contraction primitive (unit tests / micro-benchmarks)
# ---------------------------------------------------------------------------------------------------------
def gemm(A, B, *, engine="tf32", bias=None, epilogue="none", aux=None, out=None, accumulate=False, split_k=1,
         round_out=False):
    """C = epi([C +] A @ B + bias) through cfn_gemm_f32.  A (M,K) and B (K,N) are fp32 CUDA tensors with ARBITRARY
    strides (pass `.t()` views for the transposed flavours: the strides select the operand major, nothing is copied).
    engine "fp32" = CUDA-core FMA, "tf32" = tcgen05 kind::tf32 fed by TMA."""
    lib = _lib.load()
    M, K = A.shape
    K2, N = B.shape
    assert K == K2 and A.dtype == torch.float32 and B.dtype == torch.float32 and A.is_cuda and B.is_cuda
    if out is None:
        out = torch.zeros(M, N, device=A.device) if (accumulate or split_k > 1) else torch.empty(M, N, device=A.device)
    epi = {"none": 0, "relu": 1, "tanh_mask": 2, "relu_mask_mul": 3}[epilogue]
    aux_rs = aux.stride(0) if (aux is not None and aux.dim() == 2) else 0
    with torch.cuda.device(A.device):
        check(lib.cfn_gemm_f32({"fp32": 0, "tf32": 1}[engine], _ptr(A), A.stride(0), A.stride(1), _ptr(B), B.stride(0),
                               B.stride(1), _ptr(out), out.stride(0), _ptr(bias) if bias is not None else None,
                               _ptr(aux) if aux is not None else None, aux_rs, M, N, K, epi, int(accumulate), int(split_k),
                               int(round_out), _stream()), "cfn_gemm_f32")
    return out


def gemm_bf16(A, B, *, out_dtype=torch.bfloat16, bias=None, epilogue="none", aux=None, mask_out=None, aux_bits=None,
              out=None, split_k=1, rowsum=None):
    """bf16-storage flavour of `gemm` through cfn_gemm_bf16 (tcgen05 kind::f16, fp32 accumulation).  A (M,K), B (K,N)
    bf16 CUDA tensors with arbitrary strides; C bf16 or fp32.  `mask_out` / `aux_bits`: int32 (M, ceil(N/32)) ReLU bit
    masks written by epilogue "relu" / read by epilogue "relu_mask_mul"."""
    lib = _lib.load()
    M, K = A.shape
    K2, N = B.shape
    assert K == K2 and A.dtype == torch.bfloat16 and B.dtype == torch.bfloat16 and A.is_cuda
    if out is None:
        out = (torch.zeros if split_k > 1 else torch.empty)(M, N, device=A.device, dtype=out_dtype)
    epi = {"none": 0, "relu": 1, "tanh_mask": 2, "relu_mask_mul": 3}[epilogue]
    bits = mask_out if mask_out is not None else aux_bits
    with torch.cuda.device(A.device):
        check(lib.cfn_gemm_bf16(_ptr(A), A.stride(0), A.stride(1), _ptr(B), B.stride(0), B.stride(1), _ptr(out),
                                out.stride(0), int(out.dtype == torch.bfloat16), _ptr(bias) if bias is not None else None,
                                _ptr(aux) if aux is not None else None, _ptr(mask_out) if mask_out is not None else None,
                                _ptr(aux_bits) if aux_bits is not None else None, bits.stride(0) if bits is not None else 0,
                                M, N, K, epi, int(split_k), _ptr(rowsum) if rowsum is not None else None, _stream()),
              "cfn_gemm_bf16")
    return out
