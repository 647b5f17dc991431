"""F5 evaluation (cfnerf_b200.evaluate, cfn_eval_records_f32, cfn_sparsification_f32): the numpy restatement of the
metrics (tests/eval_oracle.py) on hand-checked cases; the C-ABI's host-side argument checks; and, on the GPU, the
kernels and the public calls against that restatement and the render oracle."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import eval_oracle as E
from oracle import cfnerf_oracle as O

CFN_EINVAL, CFN_ENOMEM = -1, -4


# ------------------------------------------------------------------------------------------------
# the oracle's own properties (CPU)
# ------------------------------------------------------------------------------------------------
def test_oracle_uncertainty_equal_to_error_gives_zero_rmse_ause():
    rng = np.random.default_rng(0)
    e = rng.random(500)
    r = E.sparsification(e, e, rng.random(500), 100)
    assert r["ause_rmse"] == 0.0
    assert np.array_equal(r["curves"][0], r["curves"][1])


def test_oracle_hand_computed_reversed_ranking():
    """P = 4, S = 4, uncertainty ranks the pixels exactly backwards: m = [4, 3, 2, 1]; by u the kept errors are the
    largest ones, the oracle keeps the smallest."""
    e = np.array([1.0, 2.0, 3.0, 4.0])
    r = E.sparsification(np.array([4.0, 3.0, 2.0, 1.0]), e, e, 4)
    assert np.allclose(r["fractions"], [0, 0.25, 0.5, 0.75])
    assert np.allclose(r["curves"][2], [1.0, 1.2, 1.4, 1.6]) and np.allclose(r["curves"][3], [1.0, 0.8, 0.6, 0.4])
    assert abs(r["ause_mae"] - 0.45) < 1e-12          # (1/4) * ((0 + .4) + (.4 + .8) + (.8 + 1.2)) / 2
    n = math.sqrt(2.5)
    d = [0.0, (math.sqrt(3) - math.sqrt(2)) / n, (math.sqrt(3.5) - math.sqrt(1.5)) / n, (2 - 1) / n]
    assert abs(r["ause_rmse"] - sum(0.25 * (d[i] + d[i + 1]) / 2 for i in range(3))) < 1e-12


@pytest.mark.parametrize("P", [1, 37, 1001])
def test_oracle_pixel_counts_not_divisible_by_the_fractions(P):
    rng = np.random.default_rng(P)
    u, e = rng.random(P), rng.random(P)
    r = E.sparsification(u, e, e, 100)
    m = P - (np.arange(100) * P) // 100
    assert m.min() >= 1 and m[0] == P
    order = np.argsort(u, kind="stable")
    i = 99
    want = math.sqrt(e[order][:m[i]].sum() / m[i]) / math.sqrt(e.mean())
    assert abs(r["curves"][0][i] - want) < 1e-12
    if P == 1:
        assert np.all(r["curves"] == 1.0) and r["ause_rmse"] == 0.0 and r["ause_mae"] == 0.0


def test_oracle_ties_resolved_by_pixel_index():
    u = np.zeros(4)
    e = np.array([4.0, 3.0, 2.0, 1.0])
    r = E.sparsification(u, e, e, 4)
    # stable order keeps pixels 0, 1, 2, 3: at i = 3 only pixel 0 (e = 4) is kept
    assert abs(r["curves"][2][3] - 4.0 / 2.5) < 1e-12


def test_oracle_zero_error_gives_zero_curves():
    r = E.sparsification(np.random.default_rng(1).random(50), np.zeros(50), np.zeros(50), 10)
    assert np.all(r["curves"] == 0.0) and r["ause_rmse"] == 0.0 and r["ause_mae"] == 0.0


def test_oracle_curves_start_at_one():
    rng = np.random.default_rng(2)
    r = E.sparsification(rng.random(300), rng.random(300), rng.random(300), 20)
    assert np.all(r["curves"][:, 0] == 1.0)


def test_oracle_records_follow_the_kde_nll_loss():
    g = torch.Generator().manual_seed(0)
    rgb, tgt = torch.rand(16, 3, 32, generator=g), torch.rand(16, 3, generator=g)
    rec = E.eval_records(rgb.numpy(), None, tgt.numpy(), None, 32)
    ref = O.kde_nll_loss(rgb.double(), tgt.double(), torch.tensor(0.0), 32, 0.0)
    assert abs(E.view_metrics(rec)["nll"] - float(ref["loss_nll"])) < 1e-10
    assert abs(E.view_metrics(rec)["mse"] - float(ref["mse"])) < 1e-12


# ------------------------------------------------------------------------------------------------
# C-ABI argument checks, made before any CUDA call (CPU)
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from cfnerf_b200 import _lib
    return _lib.load()


def test_sparsification_cabi_rejects_bad_arguments_on_the_host(lib):
    p = C.c_void_p(4096)

    def call(V=2, P=100, S=10, u=p, e=p, a=p, ws=p, curves=p, ause=p):
        return lib.cfn_sparsification_f32(u, e, a, V, P, S, ws, 1 << 30, curves, ause, None)

    for kw, msg in (({"V": 0}, b"n_views"), ({"P": 0}, b"n_pixels"), ({"V": -3}, b"n_views"), ({"S": 1}, b"n_fractions"),
                    ({"V": 2, "P": 1 << 30}, b"2^31"), ({"V": 1, "P": 1 << 31}, b"2^31"), ({"V": 70000}, b"65535"),
                    ({"u": None}, b"null"), ({"e": None}, b"null"), ({"a": None}, b"null"), ({"ws": None}, b"null"),
                    ({"curves": None}, b"null"), ({"ause": None}, b"null")):
        assert call(**kw) == CFN_EINVAL, kw
        assert msg in lib.cfn_last_error(), (kw, lib.cfn_last_error())
    out = C.c_size_t()
    assert lib.cfn_sparsification_workspace_bytes(0, 10, 10, C.byref(out)) == CFN_EINVAL
    assert lib.cfn_sparsification_workspace_bytes(1, 10, 1, C.byref(out)) == CFN_EINVAL
    assert lib.cfn_sparsification_workspace_bytes(1, 10, 10, None) == CFN_EINVAL
    assert lib.cfn_version() == 103


def test_eval_records_cabi_rejects_bad_arguments_on_the_host(lib):
    p = C.c_void_p(4096)
    assert lib.cfn_eval_records_f32(p, p, p, None, None, 8, 1, p, p, p, p, None, None, None, None) == CFN_EINVAL
    assert b"K >= 2" in lib.cfn_last_error()
    assert lib.cfn_eval_records_f32(p, None, p, None, None, 8, 4, p, p, p, p, None, None, None, None) == CFN_EINVAL
    assert lib.cfn_eval_records_f32(p, p, p, p, None, 8, 4, p, p, p, p, p, p, p, None) == CFN_EINVAL
    assert b"target_depth" in lib.cfn_last_error()


def test_evaluation_has_no_cpu_fallback():
    import cfnerf_b200 as cf
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    net = cf.NeRFFlowsParams(netwidth=64, K_samples=4)
    with pytest.raises(RuntimeError):
        cf.evaluate_view(O.synthetic_rays(4), torch.rand(4, 3), net)
    with pytest.raises(RuntimeError):
        cf.sparsification(torch.rand(10), torch.rand(10), torch.rand(10))


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cf():
    import cfnerf_b200
    return cfnerf_b200


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _inputs(kind, V, P, seed):
    rng = np.random.default_rng(seed)
    u, e, a = (rng.random((V, P), dtype=np.float32) for _ in range(3))
    e = e * e
    if kind == "ties":
        u = np.floor(u * 8).astype(np.float32) / 8
    elif kind == "constant":
        u = np.full((V, P), 0.25, np.float32)
    elif kind == "zero_error":
        e, a = np.zeros_like(e), np.zeros_like(a)
    return u, e, a


@pytest.mark.gpu
@pytest.mark.parametrize("V,P,S", [(1, 1, 100), (1, 37, 100), (3, 1000, 100), (1, 4096, 7), (2, 640000, 100)])
@pytest.mark.parametrize("kind", ["random", "ties", "constant", "zero_error"])
def test_sparsification_kernel_matches_the_oracle(cf, dev, V, P, S, kind):
    u, e, a = _inputs(kind, V, P, V * P + S)
    r = cf.sparsification(*(torch.from_numpy(x).to(dev) for x in (u, e, a)), n_fractions=S)
    assert tuple(r["curves"].shape) == (V, 4, S) and tuple(r["ause_rmse"].shape) == (V,)
    assert torch.equal(r["fractions"].cpu(), torch.from_numpy((np.arange(S) / S).astype(np.float32)))
    curves = r["curves"].cpu().numpy().astype(np.float64)
    for v in range(V):
        o = E.sparsification(u[v], e[v], a[v], S)
        assert np.all(np.abs(curves[v] - o["curves"]) <= 1e-6 * np.abs(o["curves"])), (v, np.abs(curves[v] - o["curves"]).max())
        assert abs(float(r["ause_rmse"][v]) - o["ause_rmse"]) <= 1e-6
        assert abs(float(r["ause_mae"][v]) - o["ause_mae"]) <= 1e-6


@pytest.mark.gpu
def test_sparsification_is_bitwise_repeatable_and_checks_its_workspace(cf, dev):
    from cfnerf_b200 import _lib
    from cfnerf_b200.engine import _ptr
    u, e, a = (torch.from_numpy(x).to(dev) for x in _inputs("ties", 3, 50000, 7))
    r1, r2 = cf.sparsification(u, e, a), cf.sparsification(u, e, a)
    assert torch.equal(r1["curves"], r2["curves"]) and torch.equal(r1["ause_rmse"], r2["ause_rmse"])
    lib = _lib.load()
    need = C.c_size_t()
    assert lib.cfn_sparsification_workspace_bytes(3, 50000, 100, C.byref(need)) == 0
    ws = torch.empty(need.value, dtype=torch.uint8, device=dev)
    curves, ause = torch.empty(3, 4, 100, device=dev), torch.empty(3, 2, device=dev)
    assert lib.cfn_sparsification_f32(_ptr(u), _ptr(e), _ptr(a), 3, 50000, 100, _ptr(ws), need.value - 1, _ptr(curves),
                                      _ptr(ause), None) == CFN_ENOMEM
    assert b"workspace" in lib.cfn_last_error()
    assert lib.cfn_sparsification_f32(_ptr(u), _ptr(e), _ptr(a), 3, 50000, 100, _ptr(ws), need.value, _ptr(curves),
                                      _ptr(ause), None) == 0
    torch.cuda.synchronize()
    assert torch.equal(curves, r1["curves"])


@pytest.mark.gpu
def test_sparsification_rejects_bad_inputs(cf, dev):
    x = torch.rand(2, 10, device=dev)
    with pytest.raises(ValueError):
        cf.sparsification(x, x[:, :5], x)
    with pytest.raises(ValueError):
        cf.sparsification(x[:, :0], x[:, :0], x[:, :0])
    with pytest.raises(ValueError):
        cf.sparsification(x, x, x, n_fractions=1)
    for bad in (-1.0, float("nan"), float("inf")):
        y = x.clone()
        y[1, 3] = bad
        with pytest.raises(ValueError):
            cf.sparsification(x, y, x)


def _small_net(cf, dev, seed=0):
    cfg = O.CfnConfig(W=256, K=64, h_alpha=32)
    p = O.make_params(cfg, seed, "lively")
    sa, sr = O.make_latents(cfg, seed)
    return cfg, p, sa, sr, cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev)


def _close(got, want, tol):
    got = np.asarray(got, np.float64)
    return float(np.max(np.abs(got - want) / np.maximum(1.0, np.abs(want))))


@pytest.mark.gpu
def test_evaluate_view_fp32_matches_the_oracle_pipeline(cf, dev):
    cfg, p, sa, sr, net = _small_net(cf, dev)
    rays = O.synthetic_rays(777, 11)
    ea, er = O.test_latents(sa, sr)
    with torch.no_grad():
        o = O.render_rays(p, cfg, rays, ea, er, False, faithful=False)
    g = torch.Generator().manual_seed(5)
    target = (o["rgb_map"].mean(-1) + 0.05 * torch.randn(777, 3, generator=g)).clamp(0, 1)
    t_depth = o["depth_map"].mean(-1) + 0.1 * torch.randn(777, generator=g)
    res = cf.evaluate_view(rays, target, net, target_depth=t_depth, precision="fp32")
    rec = E.eval_records(o["rgb_map"].numpy(), o["depth_map"].numpy(), target.numpy(), t_depth.numpy(), cfg.K)
    errs = {k: _close(res[k].cpu().numpy(), rec[k], 1e-5) for k in rec}
    print("evaluate_view fp32 vs oracle records (rel. to max(1,|x|)):", errs)
    for k, v in errs.items():
        assert v <= 1e-5, (k, v)
    m = E.view_metrics(rec)
    assert abs(res["psnr"] - m["psnr"]) <= 1e-5 * max(1.0, abs(m["psnr"])) and abs(res["nll"] - m["nll"]) <= 1e-5
    # the ordering in isolation: the oracle's sparsification of the GPU's own records
    mine = {k: res[k].cpu().numpy() for k in ("uncertainty", "sq_err", "abs_err", "depth_uncertainty", "depth_sq_err",
                                             "depth_abs_err")}
    o_rgb = E.sparsification(mine["uncertainty"], mine["sq_err"], mine["abs_err"], 100)
    o_d = E.sparsification(mine["depth_uncertainty"], mine["depth_sq_err"], mine["depth_abs_err"], 100)
    for k, want in (("ause_rmse", o_rgb["ause_rmse"]), ("ause_mae", o_rgb["ause_mae"]),
                    ("ause_depth_rmse", o_d["ause_rmse"]), ("ause_depth_mae", o_d["ause_mae"])):
        assert abs(res[k] - want) <= 1e-6, (k, res[k], want)
    assert np.all(np.abs(res["curves"].cpu().numpy() - o_rgb["curves"]) <= 1e-6 * np.abs(o_rgb["curves"]))
    assert tuple(res["rgb_mean"].shape) == (777, 3) and res["uncertainty"].is_cuda


@pytest.mark.gpu
def test_evaluate_view_fp16_stays_within_the_bar_of_the_check_mode(cf, dev):
    cfg = O.CfnConfig()
    p = O.make_params(cfg, 2, "stressed")
    sa, sr = O.make_latents(cfg, 2)
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev)
    rays = O.synthetic_rays(256, 21).to(dev)
    ks = cf.render_rays(rays, net, None, 128, False, False, precision="fp32", want_kstats=True)["kstats"]
    g = torch.Generator().manual_seed(9)
    target = (ks[:, 0:3].cpu() + 0.05 * torch.randn(256, 3, generator=g)).clamp(0, 1)
    ref = cf.evaluate_view(rays, target, net, precision="fp32")
    got = cf.evaluate_view(rays, target, net, precision="fp16")
    errs = {k: (got[k] - ref[k]).abs().max().item() for k in ("uncertainty", "sq_err", "abs_err", "nll_map")}
    print("evaluate_view fp16 vs fp32 check mode (stressed heads):", errs,
          {k: (got[k], ref[k]) for k in ("psnr", "nll", "ause_rmse", "ause_mae")})
    for k in ("uncertainty", "sq_err", "abs_err"):
        assert errs[k] <= 2e-3, (k, errs[k])


@pytest.mark.gpu
def test_evaluation_does_not_depend_on_chunking_or_batching(cf, dev):
    cfg, p, sa, sr, net = _small_net(cf, dev, 1)
    views = []
    for s in range(3):
        g = torch.Generator().manual_seed(40 + s)
        views.append((O.synthetic_rays(300, 30 + s), torch.rand(300, 3, generator=g), 3.0 + torch.rand(300, generator=g)))
    a = cf.evaluate_view(*views[0][:2], net, target_depth=views[0][2], chunk=77, precision="fp32")
    b = cf.evaluate_view(*views[0][:2], net, target_depth=views[0][2], chunk=32768, precision="fp32")
    batched = cf.evaluate_views(views, net, precision="fp32")
    singles = [a] + [cf.evaluate_view(v[0], v[1], net, target_depth=v[2], precision="fp32") for v in views[1:]]
    for x, y in [(a, b)] + list(zip(batched["views"], singles)):
        for k, v in x.items():
            if isinstance(v, torch.Tensor):
                assert torch.equal(v, y[k]), k
            else:
                assert v == y[k], (k, v, y[k])
    for k, v in batched["mean"].items():
        assert abs(v - sum(s[k] for s in singles) / 3) <= 1e-12 * max(1.0, abs(v)), k


@pytest.mark.gpu
def test_evaluate_view_coarse_fine_matches_the_oracle(cf, dev):
    cfg, pc, sa, sr, net_c = _small_net(cf, dev, 0)
    pf = O.make_params(cfg, 1, "lively")
    net_f = cf.NeRFFlowsParams.from_oracle_params(cfg, pf, sa, sr).to(dev)
    rays = O.synthetic_rays(48, 8)
    ea, er = O.test_latents(sa, sr)
    with torch.no_grad():
        o = O.render_rays_hier(pc, pf, cfg, rays, ea, er, False, 64, 128)
    g = torch.Generator().manual_seed(3)
    target = (o["rgb_map"].mean(-1) + 0.05 * torch.randn(48, 3, generator=g)).clamp(0, 1)
    res = cf.evaluate_view(rays, target, net_c, N_samples=64, N_importance=128, network_fine=net_f, precision="fp32",
                           n_fractions=10)
    rec = E.eval_records(o["rgb_map"].numpy(), None, target.numpy(), None, cfg.K)
    errs = {k: float(np.abs(res[k].cpu().numpy() - rec[k]).max()) for k in rec}
    print("coarse+fine evaluation vs oracle records:", errs)
    for k in ("uncertainty", "sq_err", "abs_err", "rgb_mean", "rgb_std"):
        assert errs[k] <= 5e-4, (k, errs[k])


@pytest.mark.gpu
def test_evaluate_view_argument_errors(cf, dev):
    net = cf.NeRFFlowsParams(netwidth=64, K_samples=1).to(dev)
    with pytest.raises(ValueError):
        cf.evaluate_view(O.synthetic_rays(4), torch.rand(4, 3), net)
    _, _, _, _, net = _small_net(cf, dev)
    with pytest.raises(ValueError):
        cf.evaluate_views([(O.synthetic_rays(4), torch.rand(4, 3)), (O.synthetic_rays(5), torch.rand(5, 3))], net)
