"""numpy fp64 restatement of the evaluation metrics cfnerf_b200.evaluate commits to (its module docstring is the
specification): per-pixel records and the sparsification curves / AUSE.  Test infrastructure only."""
import math

import numpy as np


def eval_records(rgb_map, depth_map, target, target_depth, K):
    """rgb_map (P,3,K), depth_map (P,K), target (P,3), target_depth (P) or None -> dict of per-pixel fp64 records:
    uncertainty, sq_err, abs_err, nll_map (P,), rgb_mean, rgb_std (P,3) and, with target_depth, depth_uncertainty,
    depth_sq_err, depth_abs_err."""
    x = np.asarray(rgb_map, np.float64)
    t = np.asarray(target, np.float64)
    mu = x.mean(-1)
    s = x.std(-1, ddof=1) * K / (K - 1)                                       # main:1034 / 1130
    h = (s * (0.8 / K) ** (-1.0 / 7.0) + 1e-5)[..., None]                     # main:1036
    p1 = np.exp(-((x - t[..., None]) ** 2) / (2 * h * h))
    p2 = (2 * math.pi) ** (-1.5) / h
    nll_c = -np.log((p1 * p2).mean(-1) + 1e-5)                                # main:1040-1042, per channel
    rec = {"uncertainty": (s ** 2).sum(-1) / 3, "sq_err": ((mu - t) ** 2).sum(-1) / 3,
           "abs_err": np.abs(mu - t).sum(-1) / 3, "nll_map": nll_c.sum(-1) / 3, "rgb_mean": mu, "rgb_std": s}
    if target_depth is not None:
        d = np.asarray(depth_map, np.float64)
        err = d.mean(-1) - np.asarray(target_depth, np.float64)
        rec.update(depth_uncertainty=d.var(-1, ddof=1), depth_sq_err=err ** 2, depth_abs_err=np.abs(err))
    return rec


def view_metrics(rec):
    mse = float(np.mean(rec["sq_err"]))
    return {"mse": mse, "psnr": -10.0 * math.log10(mse), "nll": float(np.mean(rec["nll_map"]))}


def _curve(x_sorted, m, root):
    cs = np.concatenate([[0.0], np.cumsum(np.asarray(x_sorted, np.float64))])
    c = cs[m] / m
    c = np.sqrt(c) if root else c
    return c / c[0] if c[0] > 0 else np.zeros_like(c)


def _ause(curve, oracle, S):
    d = curve - oracle
    return float(sum((1.0 / S) * (d[i] + d[i + 1]) / 2 for i in range(S - 1)))


def sparsification(u, e, a, S):
    """One view: u, e, a (P,) -> dict(fractions (S,), curves (4,S) [RMSE by u, RMSE oracle, MAE by u, MAE oracle],
    ause_rmse, ause_mae).  m_i = P - floor(i P / S) pixels kept, the least uncertain first (stable order: ties keep the
    lower pixel index)."""
    u, e, a = (np.asarray(v).reshape(-1) for v in (u, e, a))
    P = u.shape[0]
    i = np.arange(S, dtype=np.int64)
    m = P - (i * P) // S
    order = np.argsort(u, kind="stable")
    curves = np.stack([_curve(e[order], m, True), _curve(np.sort(e), m, True),
                       _curve(a[order], m, False), _curve(np.sort(a), m, False)])
    return {"fractions": i / S, "curves": curves, "ause_rmse": _ause(curves[0], curves[1], S),
            "ause_mae": _ause(curves[2], curves[3], S)}
