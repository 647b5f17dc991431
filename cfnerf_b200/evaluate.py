"""F5: how good is the predicted uncertainty?  PSNR, KDE-NLL and AUSE (area under the sparsification error curve) of
rendered views, computed on the device.

The reference trains CF-NeRF's K-sample predictive distribution but ships no working evaluation of it (its
`sparsification_plot`, helpers:382-438, is never called).  This module renders a held-out view chunk by chunk in test
mode, reduces every chunk to a few floats per pixel (its K fields are released right away), and runs the sparsification
of all pixels in one CUDA call.  The definitions, which this library commits to (the reference's helper is not available
to check its normalisation against), for P pixels with rgb_map (P,3,K), target t (P,3):

  mu_c, s_c    predictive mean and the reference's "uncertainty" std (unbiased std x K/(K-1), main:1034/1130), i.e.
               render_rays(..., want_kstats=True)["kstats"][:, 0:3] / [:, 3:6]
  u_p          (s_0^2 + s_1^2 + s_2^2) / 3
  e_p, a_p     mean_c (mu_c - t_c)^2 and mean_c |mu_c - t_c|
  nll_p        the KDE-NLL of main:1036-1042 averaged over the three channels
  mse, psnr    mean_p e_p and -10 log10(mse);  nll = mean_p nll_p (the trainer's loss_nll on the same maps)
  curves       for i < S: m_i = P - floor(i P / S) pixels kept, the least uncertain first (ties: lower pixel index
               first); RMSE(i) = sqrt(sum of their e / m_i), MAE(i) = sum of their a / m_i.  The oracle curves keep the
               m_i smallest errors.  Every curve is divided by its value at i = 0 (0 when that is 0).
  AUSE         sum_{i<S-1} (d_i + d_{i+1}) / (2S) with d = curve - oracle, for RMSE and MAE.
  depth        with target depth t_d: u = unbiased variance of depth over k, e / a = squared / absolute error of its
               mean; the same curves give ause_depth_rmse / ause_depth_mae.

CUDA only: without a CUDA device every call raises RuntimeError (no CPU fallback).
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib
from ._lib import check
from .api import render_rays
from .engine import _f32c, _ptr, _stream, _unwrap


def _cuda_device(what: str, t: torch.Tensor) -> torch.device:
    if not torch.cuda.is_available() or t.device.type != "cuda":
        raise RuntimeError(f"cfnerf_b200.{what} needs CUDA tensors (no CPU fallback)")
    return t.device


def _sparsify(u, e, a, n_fractions: int):
    """cfn_sparsification_f32 on (V,P) fp32 contiguous CUDA tensors -> curves (V,4,S), ause (V,2)."""
    lib = _lib.load()
    V, P = u.shape
    dev = u.device
    need = C.c_size_t()
    with torch.cuda.device(dev):
        check(lib.cfn_sparsification_workspace_bytes(V, P, n_fractions, C.byref(need)), "cfn_sparsification_workspace_bytes")
        ws = torch.empty(need.value, dtype=torch.uint8, device=dev)
        curves = torch.empty(V, 4, n_fractions, dtype=torch.float32, device=dev)
        ause = torch.empty(V, 2, dtype=torch.float32, device=dev)
        check(lib.cfn_sparsification_f32(_ptr(u), _ptr(e), _ptr(a), V, P, n_fractions, _ptr(ws), ws.numel(), _ptr(curves),
                                         _ptr(ause), _stream()), "cfn_sparsification_f32")
    return curves, ause


def _fractions(n_fractions: int, dev) -> torch.Tensor:
    return (torch.arange(n_fractions, dtype=torch.float64) / n_fractions).float().to(dev)


def sparsification(uncertainty, sq_err, abs_err, n_fractions: int = 100):
    """Sparsification curves and AUSE of one view (P,) or V views (V,P) of per-pixel uncertainty, squared error and
    absolute error (CUDA tensors, finite and >= 0).  Returns {fractions (S,), curves (V,4,S) [RMSE by uncertainty,
    RMSE oracle, MAE by uncertainty, MAE oracle], ause_rmse (V,), ause_mae (V,)}.  The input check costs one host
    sync."""
    dev = _cuda_device("sparsification", uncertainty)
    for t in (sq_err, abs_err):
        _cuda_device("sparsification", t)
    shape = tuple(uncertainty.shape)
    if tuple(sq_err.shape) != shape or tuple(abs_err.shape) != shape or len(shape) not in (1, 2):
        raise ValueError(f"uncertainty, sq_err and abs_err must share one (P,) or (V,P) shape; got "
                         f"{shape}, {tuple(sq_err.shape)}, {tuple(abs_err.shape)}")
    if shape[-1] == 0 or (len(shape) == 2 and shape[0] == 0):
        raise ValueError("sparsification needs at least one view of at least one pixel")
    if int(n_fractions) < 2:
        raise ValueError(f"n_fractions must be >= 2, got {n_fractions}")
    u, e, a = (_f32c(t, dev).reshape(-1, shape[-1]) for t in (uncertainty, sq_err, abs_err))
    bad = torch.stack([(~torch.isfinite(t)).any() | (t < 0).any() for t in (u, e, a)])
    if bool(bad.any()):
        raise ValueError("uncertainty, sq_err and abs_err must be finite and >= 0")
    curves, ause = _sparsify(u, e, a, int(n_fractions))
    return {"fractions": _fractions(int(n_fractions), dev), "curves": curves, "ause_rmse": ause[:, 0],
            "ause_mae": ause[:, 1]}


def _view_records(rays, target_rgb, target_depth, network_fn, dev, K: int, chunk: int, render_kwargs):
    """Render one view chunk by chunk and keep only the per-pixel records (device tensors of P rows)."""
    lib = _lib.load()
    P = rays.shape[0]
    t = _f32c(target_rgb, dev).reshape(P, 3)
    td = _f32c(target_depth, dev).reshape(P) if target_depth is not None else None
    f32 = dict(dtype=torch.float32, device=dev)
    rec = {k: torch.empty(P, **f32) for k in ("uncertainty", "sq_err", "abs_err", "nll_map")}
    rec["rgb_mean"], rec["rgb_std"] = torch.empty(P, 3, **f32), torch.empty(P, 3, **f32)
    if td is not None:
        for k in ("depth_uncertainty", "depth_sq_err", "depth_abs_err"):
            rec[k] = torch.empty(P, **f32)
    partial = torch.empty(min(chunk, P), 3, **f32)
    with torch.cuda.device(dev):
        for i in range(0, P, chunk):
            n = min(chunk, P - i)
            o = render_rays(_f32c(rays[i:i + n], dev), network_fn, is_train=False, want_kstats=True, **render_kwargs)
            ks, ti = o["kstats"], t[i:i + n]
            check(lib.cfn_trainer_loss_f32(_ptr(o["rgb_map"]), None, _ptr(ti), None, n, 0, K, 0.0, 0.0, _ptr(partial),
                                           None, None, _stream()), "cfn_trainer_loss_f32")
            depth = td is not None
            sl = {k: v[i:i + n] for k, v in rec.items() if v.dim() == 1}
            check(lib.cfn_eval_records_f32(_ptr(ks), _ptr(partial), _ptr(ti), _ptr(o["depth_map"] if depth else None),
                                           _ptr(td[i:i + n] if depth else None), n, K, _ptr(sl["uncertainty"]),
                                           _ptr(sl["sq_err"]), _ptr(sl["abs_err"]), _ptr(sl["nll_map"]),
                                           _ptr(sl.get("depth_uncertainty")), _ptr(sl.get("depth_sq_err")),
                                           _ptr(sl.get("depth_abs_err")), _stream()), "cfn_eval_records_f32")
            rec["rgb_mean"][i:i + n] = ks[:, 0:3]
            rec["rgb_std"][i:i + n] = ks[:, 3:6]
            del o, ks           # the chunk's K fields go back to the allocator before the next chunk renders
    return rec


def evaluate_views(views, network_fn, chunk: int = 32768, n_fractions: int = 100, **render_kwargs):
    """Evaluate several held-out views of equal pixel count: `views` is a list of (rays (P,11), target_rgb (P,3)) or
    (rays, target_rgb, target_depth (P)) tuples (all with depth targets or none).  Each view is rendered in test mode
    through `render_rays(..., want_kstats=True, **render_kwargs)` (pass N_samples=, white_bkgd=, precision=, and
    N_importance= with network_fine= for the coarse+fine model) and reduced to per-pixel records; then ONE
    cfn_sparsification_f32 call sorts all views.

    Returns {"views": [one dict per view, as evaluate_view returns], "mean": the mean over the views of psnr, mse,
    nll and every AUSE}.  The mean is taken over per-image values, which is how papers report AUSE and PSNR (not the
    metric of the pooled pixels)."""
    if not views:
        raise ValueError("evaluate_views needs at least one view")
    module = _unwrap(network_fn)
    dev = next(module.parameters()).device
    if not torch.cuda.is_available() or dev.type != "cuda":
        raise RuntimeError("cfnerf_b200.evaluate_views needs the network on a CUDA device (no CPU fallback)")
    K = int(module.K_samples)
    if K < 2:
        raise ValueError(f"evaluation needs K_samples >= 2 (unbiased std), the network has K = {K}")
    if int(n_fractions) < 2:
        raise ValueError(f"n_fractions must be >= 2, got {n_fractions}")
    P = int(views[0][0].shape[0])
    with_depth = len(views[0]) > 2 and views[0][2] is not None
    for v in views:
        if int(v[0].shape[0]) != P or int(v[1].shape[0]) != P:
            raise ValueError("every view needs the same pixel count, with one target per ray")
        if (len(v) > 2 and v[2] is not None) != with_depth:
            raise ValueError("give target depth for every view or for none")
    if P == 0:
        raise ValueError("a view needs at least one pixel")
    recs = [_view_records(v[0], v[1], v[2] if with_depth else None, network_fn, dev, K, int(chunk), render_kwargs)
            for v in views]
    keys = [("uncertainty", "sq_err", "abs_err")]
    if with_depth:
        keys.append(("depth_uncertainty", "depth_sq_err", "depth_abs_err"))
    # colour views first, then the depth views: one sort over all of them
    u, e, a = (torch.stack([r[ks[j]] for ks in keys for r in recs]) for j in range(3))
    curves, ause = _sparsify(u, e, a, int(n_fractions))
    ause = ause.double().cpu()
    fractions = _fractions(int(n_fractions), dev)
    V = len(views)
    out = []
    for i, r in enumerate(recs):
        mse = r["sq_err"].double().mean().item()
        res = {"psnr": -10.0 * math.log10(mse) if mse > 0 else math.inf, "mse": mse,
               "nll": r["nll_map"].double().mean().item(),
               "ause_rmse": float(ause[i, 0]), "ause_mae": float(ause[i, 1]), "curves": curves[i], "fractions": fractions}
        if with_depth:
            res.update(ause_depth_rmse=float(ause[V + i, 0]), ause_depth_mae=float(ause[V + i, 1]),
                       depth_curves=curves[V + i])
        res.update(r)
        out.append(res)
    scalars = ["psnr", "mse", "nll", "ause_rmse", "ause_mae"] + (["ause_depth_rmse", "ause_depth_mae"] if with_depth else [])
    return {"views": out, "mean": {k: sum(o[k] for o in out) / V for k in scalars}}


def evaluate_view(rays, target_rgb, network_fn, target_depth=None, chunk: int = 32768, n_fractions: int = 100,
                  **render_kwargs):
    """PSNR, KDE-NLL and AUSE of one held-out view.  rays (P,11) on the host or the device, target_rgb (P,3),
    optional target_depth (P).  The view is rendered in test mode, `chunk` rays at a time, through
    `render_rays(..., want_kstats=True, **render_kwargs)`; only a few floats per pixel are kept.

    Returns psnr, mse, nll, ause_rmse, ause_mae (python floats; ause_depth_rmse / ause_depth_mae and depth_curves with
    target depth), curves (4,S) [RMSE by uncertainty, RMSE oracle, MAE by uncertainty, MAE oracle], fractions (S,),
    and the per-pixel device maps uncertainty, sq_err, abs_err, nll_map (P,), rgb_mean, rgb_std (P,3) — the
    `heatmap_mse` / `heatmap_v` images of main:1143-1147 once reshaped to (H,W).  The module docstring defines every
    metric."""
    view = (rays, target_rgb) if target_depth is None else (rays, target_rgb, target_depth)
    return evaluate_views([view], network_fn, chunk=chunk, n_fractions=n_fractions, **render_kwargs)["views"][0]
