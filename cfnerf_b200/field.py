"""F6: the radiance field's K-sample distribution at 3-D points — density and colour mean / std per point and on grids,
reduced over the latent draws on the device.

CF-NeRF learns a distribution over radiance fields: every 3-D point x (with view direction d) carries K latent draws
pushed through the two conditional flow stacks, giving raw values (z0_k, z1_k, z2_k, za_k) — exactly the `raw` that
`run_network` returns for that point.  Per point this module returns 8 fp32 values

  [sigma_mean, sigma_std, r_mean, g_mean, b_mean, r_std, g_std, b_std]

  sigma_k      softplus(za_k), the reference's density activation (main:424)
  c_k          sigmoid(z_k) per channel, its colour activation (main:431)
  mean         (1/K) sum_k x_k
  std          sqrt(sum_k (x_k - mean)^2 / (K - 1)), and 0 when K = 1

The std is the plain sample std.  It is NOT the pixel "uncertainty" of `render_rays(..., want_kstats=True)`, which
carries the reference's extra K/(K-1) factor (main:1034), a pixel-level convention.  Density does not depend on the view
direction (the alpha flow parameters come from the trunk, before the view branch); colour does.

The latent draws default to the test-mode draws (`api.test_latents`: constructor-time, the last one zeroed), the draws a
test-mode render uses; eps_alpha (K,1) / eps_rgb (K,3) replace them.  Points are taken in the model's input space (no NDC
conversion) and view directions are used as given: normalise them as `render` does (main:136-144).

The network stage (K1, `cfn_network_fwd` with explicit points) writes each point's 18F flow record once; the stats kernel
(`cfn_field_stats_f32`) runs both flow stacks for all K draws and keeps 32 bytes per point, so the (M,K,4) raw samples
(16 K bytes per point: 34 GB for a 256^3 grid at K = 128) never exist.  Points are processed `chunk` at a time and each
chunk's records are released before the next one is computed.

For the coarse+fine model, query each network separately: pass `network_fine` as `network_fn` for the fine field.

CUDA only: without a CUDA device every call raises RuntimeError (no CPU fallback).
"""
from __future__ import annotations

import torch

from . import api
from .engine import _f32c, _unwrap, engine_for

# the render path's K1 launch size: 4 194 304 points = 1.2 GB of flow records at F = 4
DEFAULT_CHUNK = 1 << 22


def _cuda_module(what: str, network_fn):
    module = _unwrap(network_fn)
    dev = next(module.parameters()).device
    if not torch.cuda.is_available() or dev.type != "cuda":
        raise RuntimeError(f"cfnerf_b200.{what} needs the network on a CUDA device (no CPU fallback)")
    return module, dev


def _draws(module, K: int, dev, eps_alpha, eps_rgb):
    """-> eps_a (K), eps_c (K,3) fp32 contiguous on dev; the test-mode draws when neither is given."""
    if eps_alpha is None and eps_rgb is None:
        return api.test_latents(module, dev)
    if eps_alpha is None or eps_rgb is None:
        raise ValueError("pass both eps_alpha (K,1) and eps_rgb (K,3), or neither")
    if tuple(eps_alpha.shape) not in ((K, 1), (K,)):
        raise ValueError(f"eps_alpha must be (K,1) = ({K},1), got {tuple(eps_alpha.shape)}")
    if tuple(eps_rgb.shape) != (K, 3):
        raise ValueError(f"eps_rgb must be (K,3) = ({K},3), got {tuple(eps_rgb.shape)}")
    return _f32c(eps_alpha.reshape(K), dev), _f32c(eps_rgb, dev)


def _check_chunk(chunk) -> int:
    chunk = int(chunk)
    if chunk < 1:
        raise ValueError(f"chunk must be >= 1, got {chunk}")
    return chunk


def _run(network_fn, dev, M: int, points, viewdir_rows, chunk: int, precision, eps_a, eps_c):
    """Network stage + stats kernel over [0, M) in chunks; points(i, n) / viewdir_rows(i, n) give the (n,3) fp32
    contiguous device rows of the chunk starting at i.  -> stats (M,8)."""
    eng = engine_for(network_fn, dev, precision or api.DEFAULT_PRECISION)
    stats = torch.empty(M, 8, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev), torch.no_grad():
        for i in range(0, M, chunk):
            n = min(chunk, M - i)
            fp = eng.network(n, 1, pts=points(i, n), viewdirs=viewdir_rows(i, n))
            eng.field_stats(fp, eps_a, eps_c, out=stats[i:i + n])
            del fp              # the chunk's flow records go back to the allocator before the next chunk
    return stats


def _views(stats: torch.Tensor, shape) -> dict:
    s = stats.reshape(*shape, 8)
    return {"stats": s, "sigma_mean": s[..., 0], "sigma_std": s[..., 1], "rgb_mean": s[..., 2:5], "rgb_std": s[..., 5:8]}


def query_field(pts, network_fn, viewdirs, *, chunk: int = DEFAULT_CHUNK, precision=None, eps_alpha=None, eps_rgb=None):
    """Density and colour statistics over the K latent draws at M points (module docstring: definitions).

    pts (M,3) and viewdirs (M,3), or viewdirs (3,) for one direction shared by every point, on the host or the device
    (used as given: normalise directions first).  `precision` selects the network stage's mode like `render_rays` (default:
    the render default, fp16); the flow math follows it as K2's does.  Returns {"stats" (M,8), "sigma_mean" (M,),
    "sigma_std" (M,), "rgb_mean" (M,3), "rgb_std" (M,3)}, the last four views of "stats", on the network's device."""
    module, dev = _cuda_module("query_field", network_fn)
    if pts.dim() != 2 or pts.shape[1] != 3:
        raise ValueError(f"pts must be (M,3), got {tuple(pts.shape)}")
    M = int(pts.shape[0])
    shared_dir = tuple(viewdirs.shape) == (3,)
    if not shared_dir and tuple(viewdirs.shape) != (M, 3):
        raise ValueError(f"viewdirs must be (M,3) = ({M},3) or (3,), got {tuple(viewdirs.shape)}")
    chunk = _check_chunk(chunk)
    eps_a, eps_c = _draws(module, int(module.K_samples), dev, eps_alpha, eps_rgb)
    if shared_dir:
        vd = _f32c(viewdirs, dev).reshape(1, 3)
        vrows = lambda i, n: vd.expand(n, 3).contiguous()                # noqa: E731
    else:
        vrows = lambda i, n: _f32c(viewdirs[i:i + n], dev)                # noqa: E731
    stats = _run(network_fn, dev, M, lambda i, n: _f32c(pts[i:i + n], dev), vrows, chunk, precision, eps_a, eps_c)
    return _views(stats, (M,))


def field_grid(network_fn, bounds, resolution, viewdir=(0., 0., -1.), **query_kwargs):
    """query_field on the Rx x Ry x Rz grid spanning `bounds` = ((x0,x1),(y0,y1),(z0,z1)); `resolution` is an int or a
    3-tuple.  The axes are torch.linspace(lo, hi, R) (fp32, computed on the device) and the points are their
    meshgrid(indexing="ij"): point [i,j,k] = (xs[i], ys[j], zs[k]).  The points are generated on the device one chunk at a
    time, so the (R^3,3) point array never exists.  `viewdir` (3,) is shared by every point.  query_kwargs: chunk,
    precision, eps_alpha, eps_rgb as for query_field.

    Returns the keys of query_field shaped (Rx,Ry,Rz) / (Rx,Ry,Rz,3) ("stats": (Rx,Ry,Rz,8)), plus "axes": (xs, ys, zs)."""
    module, dev = _cuda_module("field_grid", network_fn)
    res = (int(resolution),) * 3 if isinstance(resolution, int) else tuple(int(r) for r in resolution)
    if len(res) != 3 or min(res) < 1:
        raise ValueError(f"resolution must be an int or a 3-tuple of ints >= 1, got {resolution}")
    bounds = [tuple(float(v) for v in b) for b in bounds]
    if len(bounds) != 3 or any(len(b) != 2 for b in bounds):
        raise ValueError(f"bounds must be ((x0,x1),(y0,y1),(z0,z1)), got {bounds}")
    unknown = set(query_kwargs) - {"chunk", "precision", "eps_alpha", "eps_rgb"}
    if unknown:
        raise TypeError(f"field_grid got unexpected keyword arguments {sorted(unknown)}")
    chunk = _check_chunk(query_kwargs.get("chunk", DEFAULT_CHUNK))
    eps_a, eps_c = _draws(module, int(module.K_samples), dev, query_kwargs.get("eps_alpha"), query_kwargs.get("eps_rgb"))
    vd = torch.as_tensor(viewdir, dtype=torch.float32)
    if tuple(vd.shape) != (3,):
        raise ValueError(f"viewdir must be (3,), got {tuple(vd.shape)}")
    vd = vd.to(dev).reshape(1, 3)
    Rx, Ry, Rz = res
    axes = tuple(torch.linspace(lo, hi, R, dtype=torch.float32, device=dev) for (lo, hi), R in zip(bounds, res))
    xs, ys, zs = axes

    def points(i, n):
        j = torch.arange(i, i + n, device=dev)
        return torch.stack([xs[j // (Ry * Rz)], ys[(j // Rz) % Ry], zs[j % Rz]], -1)

    stats = _run(network_fn, dev, Rx * Ry * Rz, points, lambda i, n: vd.expand(n, 3).contiguous(), chunk,
                 query_kwargs.get("precision"), eps_a, eps_c)
    out = _views(stats, res)
    out["axes"] = axes
    return out
