"""F6 field-space statistics (cfnerf_b200.field, cfn_field_stats_f32): the fp64 numpy restatement of the definitions on
hand-checked cases and the C-ABI's host-side argument checks (CPU); on the GPU the kernel against the oracle's
run_network, against the library's own run_network at the same precision, its invariances, the grid surface, the edge
cases and a full-size grid's memory."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import cfnerf_oracle as O

CFN_EINVAL, CFN_ESTATE = -1, -3


def field_stats_ref(raw):
    """The definitions of cfnerf_b200/field.py restated in fp64: raw (M,K,4) [rgb|sigma] -> (M,8) [sigma mean, sigma
    std, rgb mean (3), rgb std (3)], std = sample std with 1/(K-1), 0 when K = 1."""
    raw = np.asarray(raw, np.float64)
    K = raw.shape[1]
    za = raw[..., 3]
    sigma = np.where(za > 20.0, za, np.log1p(np.exp(np.minimum(za, 20.0))))     # F.softplus(beta=1, threshold=20)
    x = np.concatenate([sigma[..., None], 1.0 / (1.0 + np.exp(-raw[..., 0:3]))], -1)   # (M,K,4)
    m = x.mean(1)
    s = np.sqrt(((x - m[:, None]) ** 2).sum(1) / (K - 1)) if K > 1 else np.zeros_like(m)
    return np.stack([m[:, 0], s[:, 0], m[:, 1], m[:, 2], m[:, 3], s[:, 1], s[:, 2], s[:, 3]], -1)


# ------------------------------------------------------------------------------------------------
# the restatement's own properties (CPU)
# ------------------------------------------------------------------------------------------------
def test_reference_single_draw_has_zero_std():
    r = field_stats_ref(np.random.default_rng(0).normal(size=(5, 1, 4)))
    assert np.all(r[:, [1, 5, 6, 7]] == 0.0)


def test_reference_identical_draws_have_zero_std():
    raw = np.repeat(np.random.default_rng(1).normal(size=(7, 1, 4)), 16, axis=1)
    assert np.all(np.abs(field_stats_ref(raw)[:, [1, 5, 6, 7]]) <= 1e-15)


def test_reference_means_of_constant_raw_values():
    raw = np.broadcast_to(np.array([0.3, -1.2, 2.0, 0.7]), (3, 8, 4))
    r = field_stats_ref(raw)
    assert np.allclose(r[:, 0], np.log1p(np.exp(0.7)), rtol=0, atol=1e-15)
    assert np.allclose(r[:, 2:5], 1.0 / (1.0 + np.exp(-np.array([0.3, -1.2, 2.0]))), rtol=0, atol=1e-15)
    big = field_stats_ref(np.full((1, 2, 4), 30.0))
    assert big[0, 0] == 30.0                                                    # softplus threshold (main:424)


def test_reference_std_is_the_plain_sample_std():
    raw = np.zeros((1, 4, 4))
    raw[0, :, 0] = [-1.0, 0.0, 1.0, 2.0]
    c = 1.0 / (1.0 + np.exp(-raw[0, :, 0]))
    assert abs(field_stats_ref(raw)[0, 5] - np.std(c, ddof=1)) <= 1e-15


# ------------------------------------------------------------------------------------------------
# C-ABI argument checks, made before any CUDA call (CPU)
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from cfnerf_b200 import _lib
    return _lib.load()


def test_field_stats_cabi_rejects_a_null_handle_on_the_host(lib):
    p = C.c_void_p(4096)
    assert lib.cfn_field_stats_f32(None, p, p, p, 10, p, None) == CFN_EINVAL
    assert b"null handle" in lib.cfn_last_error()
    assert lib.cfn_field_stats_f32(None, None, None, None, 0, None, None) == CFN_EINVAL
    assert lib.cfn_version() == 103          # the feature is detected by the symbol, not by the version


def test_field_queries_have_no_cpu_fallback():
    import cfnerf_b200 as cf
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    net = cf.NeRFFlowsParams(netwidth=64, K_samples=4)
    with pytest.raises(RuntimeError):
        cf.query_field(torch.rand(10, 3), net, torch.tensor([0.0, 0.0, -1.0]))
    with pytest.raises(RuntimeError):
        cf.field_grid(net, ((-1, 1), (-1, 1), (-1, 1)), 4)


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


def _net(cf, dev, cfg, seed, variant):
    p = O.make_params(cfg, seed, variant)
    sa, sr = O.make_latents(cfg, seed)
    return p, sa, sr, cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev)


def _points(M, seed, scale=1.5):
    g = torch.Generator().manual_seed(seed)
    pts = (torch.rand(M, 3, generator=g) * 2 - 1) * scale
    dirs = torch.nn.functional.normalize(torch.randn(M, 3, generator=g), dim=-1)
    return pts, dirs


def _oracle_stats(p, cfg, pts, dirs, ea, er, dtype, block=8192):
    """oracle.run_network in `dtype` (test mode, the cheap conditioning path), reduced in fp64, in blocks of points."""
    pd = {k: v.to(dtype) for k, v in p.items()}
    out = []
    with torch.no_grad():
        for i in range(0, pts.shape[0], block):
            raw, _ = O.run_network(pd, cfg, pts[i:i + block, None].to(dtype), dirs[i:i + block].to(dtype), ea.to(dtype),
                                   er.to(dtype), False, faithful=False)
            out.append(field_stats_ref(raw[:, 0].numpy()))
    return np.concatenate(out)


def _rel(got, want):
    got = np.asarray(got, np.float64)
    return np.abs(got - want) / np.maximum(1.0, np.abs(want))


# (variant, K, F, M, custom draws): both weight variants, K in {1, 16, 32, 40, 128}, F = 4 (compile-time) and the
# runtime-F instantiation (F = 2, 8), M in {1, 37, 100 003}, the test-mode draws and caller-given draws
ORACLE_CASES = [("lively", 1, 4, 37, False), ("lively", 16, 2, 37, True), ("stressed", 32, 4, 100003, False),
                ("stressed", 40, 8, 37, True), ("lively", 128, 4, 1, False), ("stressed", 128, 2, 1000, False),
                ("lively", 40, 4, 1000, True), ("stressed", 16, 8, 1, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("variant,K,F,M,custom", ORACLE_CASES)
def test_fp32_check_mode_matches_the_oracle(cf, dev, variant, K, F, M, custom):
    cfg = O.CfnConfig(W=128, K=K, F=F)
    p, sa, sr, net = _net(cf, dev, cfg, K + F, variant)
    pts, dirs = _points(M, M + K)
    if custom:
        g = torch.Generator().manual_seed(77)
        ea, er = torch.randn(K, 1, generator=g), torch.randn(K, 3, generator=g)
        got = cf.query_field(pts, net, dirs, precision="fp32", eps_alpha=ea, eps_rgb=er)
    else:
        ea, er = O.test_latents(sa, sr)
        got = cf.query_field(pts, net, dirs, precision="fp32")
    s = got["stats"].cpu().numpy()
    ref64 = _oracle_stats(p, cfg, pts, dirs, ea, er, torch.float64)
    ref32 = _oracle_stats(p, cfg, pts, dirs, ea, er, torch.float32)
    # conditioning-aware bar, as for the network stage (test_gpu_parity): the stressed heads amplify fp32 rounding, so the
    # bar is the larger of 1e-5 and three times the oracle's own fp32-vs-fp64 distance
    noise = float(_rel(ref32, ref64).max())
    err = _rel(s, ref64).max(0)
    tol = max(1e-5, 3 * noise)
    print(f"{variant} K={K} F={F} M={M} custom={custom}: max rel err per output {np.array2string(err, precision=2)}, "
          f"oracle fp32 noise {noise:.2e}, bar {tol:.2e}")
    assert s.shape == (M, 8) and float(err.max()) <= tol
    if K == 1:
        assert np.all(s[:, [1, 5, 6, 7]] == 0.0)
    assert torch.equal(got["sigma_mean"], got["stats"][:, 0]) and torch.equal(got["rgb_std"], got["stats"][:, 5:8])


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["lively", "stressed"])
def test_tensor_core_modes_against_the_fp32_check_mode(cf, dev, variant):
    """Per-point statistics in the tensor-core modes against the fp32 check mode, relative to max(1, |ref|), over 20 000
    points of the canonical network.  What differs is the network stage's operand precision (the stats kernel itself
    follows K2 to ~4e-7, test_same_precision_as_run_network_reduced_on_the_host).  A rendered pixel averages many
    samples; a single point does not, so on the stressed heads (SURVEY §8(d)) the 2e-3 render bar holds for 99 % of the
    points and the worst point is pinned at its measured level (fp16 1.35e-2, tf32 1.05e-2 on a B200).  bf16 operands
    are outside the bar on that fixture, as for rendering, and pinned too (p99 2e-2, worst 9e-2).  On the lively weights
    fp16 and tf32 keep every point inside the bar (worst 5e-5)."""
    cfg = O.CfnConfig(K=32)
    _, _, _, net = _net(cf, dev, cfg, 2, variant)
    pts, dirs = _points(20000, 3)
    ref = cf.query_field(pts, net, dirs, precision="fp32")["stats"].double()
    errs = {}
    for prec in ("fp16", "tf32", "bf16"):
        s = cf.query_field(pts, net, dirs, precision=prec)["stats"].double()
        e = ((s - ref).abs() / ref.abs().clamp_min(1.0)).cpu().numpy()
        errs[prec] = {"max": float(e.max()), "p99": float(np.quantile(e, 0.99, axis=0).max()), "mean": float(e.mean())}
    print(f"field stats vs the fp32 check mode ({variant}):", errs)
    if variant == "lively":
        for prec in ("fp16", "tf32"):
            assert errs[prec]["max"] <= 2e-3, (prec, errs[prec])
        assert errs["bf16"]["max"] <= 1e-2, errs["bf16"]
        return
    for prec in ("fp16", "tf32"):
        assert errs[prec]["p99"] <= 2e-3 and errs[prec]["max"] <= 2e-2, (prec, errs[prec])
    assert errs["bf16"]["p99"] <= 5e-2 and errs["bf16"]["max"] <= 0.15, errs["bf16"]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp16", "fp32"])
@pytest.mark.parametrize("variant", ["lively", "stressed"])
def test_same_precision_as_run_network_reduced_on_the_host(cf, dev, precision, variant):
    """Pins the stats kernel's flow math to K2's: the raw samples of run_network (K2) at the same precision, reduced in
    fp64 on the host, against query_field."""
    cfg = O.CfnConfig(W=256, K=40, h_alpha=32)
    _, _, _, net = _net(cf, dev, cfg, 4, variant)
    pts, dirs = _points(5000, 9)
    raw, _ = cf.run_network(pts.to(dev)[:, None, :], dirs.to(dev), net, False, True, precision=precision)
    ref = field_stats_ref(raw[:, 0].cpu().numpy())
    got = cf.query_field(pts, net, dirs, precision=precision)["stats"].cpu().numpy()
    err = _rel(got, ref).max(0)
    print(f"{variant}[{precision}] query_field vs run_network + fp64 reduction: {np.array2string(err, precision=2)}")
    assert float(err.max()) <= 2e-6


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_bitwise_invariances(cf, dev, precision):
    cfg = O.CfnConfig(W=256, K=32, h_alpha=32)
    _, _, _, net = _net(cf, dev, cfg, 5, "lively")
    pts, dirs = _points(10007, 11)
    pts = pts.to(dev)
    a = cf.query_field(pts, net, dirs.to(dev), precision=precision)["stats"]
    b = cf.query_field(pts, net, dirs.to(dev), precision=precision)["stats"]
    c = cf.query_field(pts, net, dirs.to(dev), precision=precision, chunk=1000)["stats"]
    assert torch.equal(a, b) and torch.equal(a, c)
    # a point's result does not depend on the other points of the call
    assert torch.equal(cf.query_field(pts[5000:5001], net, dirs[5000:5001].to(dev), precision=precision)["stats"][0], a[5000])
    # density does not depend on the view direction; colour does
    other = cf.query_field(pts, net, torch.tensor([0.0, 0.6, -0.8], device=dev), precision=precision)["stats"]
    assert torch.equal(other[:, 0:2], a[:, 0:2])
    assert not torch.equal(other[:, 2:5], a[:, 2:5])


@pytest.mark.gpu
def test_field_grid_equals_query_field_on_the_meshgrid(cf, dev):
    cfg = O.CfnConfig(W=128, K=16)
    _, _, _, net = _net(cf, dev, cfg, 6, "lively")
    bounds = ((-1.0, 0.5), (0.2, 1.9), (-0.7, -0.1))
    vdir = (0.6, 0.0, -0.8)
    g = cf.field_grid(net, bounds, (5, 7, 3), viewdir=vdir, precision="fp32", chunk=17)
    assert tuple(g["stats"].shape) == (5, 7, 3, 8) and tuple(g["sigma_mean"].shape) == (5, 7, 3)
    assert tuple(g["rgb_mean"].shape) == (5, 7, 3, 3) and tuple(g["rgb_std"].shape) == (5, 7, 3, 3)
    xs, ys, zs = g["axes"]
    for ax, (lo, hi), R in zip(g["axes"], bounds, (5, 7, 3)):
        assert torch.equal(ax, torch.linspace(lo, hi, R, dtype=torch.float32, device=dev))
    X, Y, Z = torch.meshgrid(xs, ys, zs, indexing="ij")
    pts = torch.stack([X, Y, Z], -1).reshape(-1, 3)
    q = cf.query_field(pts, net, torch.tensor(vdir), precision="fp32")
    assert torch.equal(g["stats"].reshape(-1, 8), q["stats"])
    # 'ij' order: [i, j, k] is the point (xs[i], ys[j], zs[k])
    one = cf.query_field(torch.stack([xs[4], ys[1], zs[2]])[None], net, torch.tensor(vdir), precision="fp32")["stats"][0]
    assert torch.equal(g["stats"][4, 1, 2], one)
    assert torch.equal(cf.field_grid(net, bounds, (5, 7, 3), viewdir=vdir, precision="fp32")["stats"], g["stats"])


@pytest.mark.gpu
def test_edge_cases_and_argument_errors(cf, dev):
    from cfnerf_b200 import _lib
    from cfnerf_b200.engine import _ptr
    cfg = O.CfnConfig(W=128, K=8)
    _, _, _, net = _net(cf, dev, cfg, 7, "lively")
    vd = torch.tensor([0.0, 0.0, -1.0])
    cf.query_field(torch.rand(4, 3), net, vd)                   # engine created, weights packed
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        r = cf.query_field(torch.empty(0, 3), net, vd)
        torch.cuda.synchronize()
    assert tuple(r["stats"].shape) == (0, 8) and tuple(r["rgb_mean"].shape) == (0, 3) and r["stats"].is_cuda
    kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
               and "memcpy" not in e.name.lower() and "memset" not in e.name.lower()]
    assert not kernels, kernels
    pts = torch.rand(10, 3)
    for kw in ({"eps_alpha": torch.zeros(7, 1), "eps_rgb": torch.zeros(8, 3)},
               {"eps_alpha": torch.zeros(8, 1), "eps_rgb": torch.zeros(8, 2)},
               {"eps_alpha": torch.zeros(8, 1)}):
        with pytest.raises(ValueError):
            cf.query_field(pts, net, vd, **kw)
    for bad in (torch.zeros(9, 3), torch.zeros(10, 2), torch.zeros(2)):
        with pytest.raises(ValueError):
            cf.query_field(pts, net, bad)
    with pytest.raises(ValueError):
        cf.query_field(torch.rand(10, 2), net, vd)
    with pytest.raises(ValueError):
        cf.field_grid(net, ((0, 1), (0, 1), (0, 1)), (4, 0, 4))
    # the C-ABI on a handle whose weights were never packed, and its argument checks
    lib = _lib.load()
    c = _lib.CfnConfigC(D=cfg.D, W=cfg.W, L_pos=cfg.L_pos, L_dir=cfg.L_dir, h_alpha=cfg.h_alpha, h_rgb=cfg.h_rgb, F=cfg.F,
                        K=cfg.K, precision=_lib.PREC["fp32"])
    h = C.c_void_p()
    _lib.check(lib.cfn_create(C.byref(c), C.byref(h)), "cfn_create")
    try:
        buf = torch.zeros(64, 72, device=dev)
        p = _ptr(buf)
        assert lib.cfn_field_stats_f32(h, p, p, p, 4, p, None) == CFN_ESTATE
        assert b"cfn_pack_weights first" in lib.cfn_last_error()
        assert lib.cfn_field_stats_f32(h, p, p, p, -1, p, None) == CFN_EINVAL
        assert lib.cfn_field_stats_f32(h, p, None, p, 4, p, None) == CFN_EINVAL
        assert b"null" in lib.cfn_last_error()
    finally:
        lib.cfn_destroy(h)
    eng = cf.engine_for(net, dev, "fp16")
    eng.pack()
    assert lib.cfn_field_stats_f32(eng.h, None, None, None, 0, None, None) == 0


@pytest.mark.gpu
def test_a_256_cubed_grid_at_k128_stays_within_one_chunk_of_memory(cf, dev):
    cfg = O.CfnConfig(K=128)
    _, _, _, net = _net(cf, dev, cfg, 0, "default")
    R, chunk = 256, 1 << 22
    M = R ** 3
    cf.field_grid(net, ((-1, 1),) * 3, 4)                       # engine created, weights packed
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    g = cf.field_grid(net, ((-1.5, 1.5),) * 3, R, chunk=chunk)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated(dev) - base
    # one chunk's flow records + the (M,8) outputs + one chunk of points, directions and index temporaries (< 96 B per
    # point) + 64 MB; the K1 workspace of the tensor-core modes is 256 bytes
    bound = chunk * 18 * cfg.F * 4 + M * 32 + chunk * 96 + (64 << 20)
    print(f"256^3 grid at K=128: peak {peak / 2**30:.2f} GiB, bound {bound / 2**30:.2f} GiB, raw samples would be "
          f"{M * cfg.K * 16 / 2**30:.1f} GiB")
    assert peak <= bound < 4 << 30
    s = g["stats"]
    assert tuple(s.shape) == (R, R, R, 8) and bool(torch.isfinite(s).all())
    assert bool((s[..., [1, 5, 6, 7]] >= 0).all()) and bool(((s[..., 2:5] >= 0) & (s[..., 2:5] <= 1)).all())
