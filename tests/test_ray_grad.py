"""F7 on the GPU: gradients with respect to the ray record and the camera pose.

fp32 check mode against the oracle's autograd (float32 on the CPU) in train and test mode, the tensor-core chains
against fp32, the pose adjoint, bitwise repeatability, the frozen-network path, and an end-to-end pose refinement."""
import math

import pytest
import torch

from oracle import cfnerf_oracle as O

pytestmark = pytest.mark.gpu

GROUPS = {"o": slice(0, 3), "d": slice(3, 6), "near/far": slice(6, 8), "viewdir": slice(8, 11)}
CFG = dict(D=4, W=64, L_pos=10, L_dir=4, h_alpha=16, h_rgb=16, F=4)


@pytest.fixture(scope="module")
def cf():
    import cfnerf_b200
    return cfnerf_b200


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def _rel(a, b):
    return (a.double().cpu() - b.double().cpu()).norm().item() / max(b.double().norm().item(), 1e-30)


def _setup(K, B, n_depth, perturb, seed=3, W=64):
    cfg = O.CfnConfig(K=K, **dict(CFG, W=W))
    p = O.make_params(cfg, seed, "lively")
    sa, sr = O.make_latents(cfg, seed)
    g = torch.Generator().manual_seed(seed + 10)
    rays = O.synthetic_rays(B, seed + 1, near=2.0, far=6.0)
    rays[:, 3:6] *= (0.7 + 0.6 * torch.rand(B, 1, generator=g))      # |d| != 1
    t_rand = torch.rand(B, 128, generator=g) if perturb else None
    target = torch.rand(B - n_depth, 3, generator=g)
    td = (3.0 + torch.rand(n_depth, generator=g)) if n_depth else None
    return cfg, p, sa, sr, rays, t_rand, target, td, g


def _library_grads(cf, dev, cfg, p, sa, sr, rays, train, t_rand, target, td, eps, precision, lindisp, white_bkgd,
                   netchunk, params_grad=True):
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev)
    net.requires_grad_(params_grad)
    r = rays.to(dev).requires_grad_(True)
    kw = dict(eps_alpha=eps[0].to(dev), eps_rgb=eps[1].to(dev)) if train else {}
    out = cf.render_rays(r, net, None, 128, train, False, K_samples=cfg.K, perturb=1. if t_rand is not None else 0.,
                         t_rand=t_rand.to(dev) if t_rand is not None else None, precision=precision, lindisp=lindisp,
                         white_bkgd=white_bkgd, netchunk=netchunk, **kw)
    if not train:
        out = dict(out, loss_entropy=torch.zeros(1, 1, 1, device=dev))
    res = cf.trainer_loss(out, target.to(dev), cfg.K, 0.01 if train else 0.0,
                          target_depth=td.to(dev) if td is not None else None, depth_lambda=0.5)
    res["loss"].backward()
    torch.cuda.synchronize()
    return r.grad.detach().cpu(), {n: q.grad for n, q in net.named_parameters()}


def _oracle_grads(cfg, p, sa, sr, rays, train, t_rand, target, td, eps, lindisp, white_bkgd, netchunk):
    pr = {k: v.clone().requires_grad_(True) for k, v in p.items()}
    r = rays.clone().requires_grad_(True)
    ea, er = eps if train else O.test_latents(sa, sr)
    out = O.render_rays(pr, cfg, r, ea, er, train, t_rand=t_rand, lindisp=lindisp, white_bkgd=white_bkgd,
                        faithful=False, netchunk=netchunk)
    if train:
        loss = O.trainer_loss(out, target, cfg.K, 0.01, target_depth=td, depth_lambda=0.5)["loss"]
    else:
        nb = target.shape[0]
        loss = O.kde_nll_loss(out["rgb_map"][:nb], target, 0.0, cfg.K, 0.0)["loss"]
        if td is not None:
            loss = loss + 0.5 * torch.mean((out["depth_map"].mean(-1)[nb:] - td) ** 2)
    loss.backward()
    return r.grad, {k: v.grad for k, v in pr.items()}


# (train, K, B, depth rays, perturb, lindisp, white_bkgd, netchunk): B = 1 / 37 / 700 / 1600 rays; several latent groups
# where netchunk < 128 B (train mode draws one latent pair per group)
CASES = [
    (True, 16, 37, 7, True, False, True, 65536),
    (True, 32, 700, 100, True, True, False, 128 * 256),
    (True, 40, 1600, 0, False, False, True, 128 * 512),
    (True, 16, 1, 0, True, False, False, 65536),
    (False, 16, 37, 0, True, True, True, 65536),
    (False, 32, 700, 100, False, False, False, 65536),
    (False, 40, 1600, 200, True, False, True, 65536),
    (False, 32, 1, 0, False, True, False, 65536),
]


@pytest.mark.parametrize("train,K,B,n_depth,perturb,lindisp,white_bkgd,netchunk", CASES)
def test_fp32_ray_gradient_vs_oracle_autograd(cf, dev, train, K, B, n_depth, perturb, lindisp, white_bkgd, netchunk):
    """ray_batch.grad after render_rays + trainer_loss backward, fp32 check mode, against the oracle's autograd: relative
    L2 distance per column group within 2e-3 (the repository's gradient bar); the parameter gradients of the same call
    keep their bar."""
    cfg, p, sa, sr, rays, t_rand, target, td, g = _setup(K, B, n_depth, perturb)
    G = max(1, math.ceil(B * 128 / netchunk)) if train else 1
    eps = (torch.randn(G, K, 1, generator=g), torch.randn(G, K, 3, generator=g))
    if G == 1:
        eps = (eps[0][0], eps[1][0])
    gr, gp = _library_grads(cf, dev, cfg, p, sa, sr, rays, train, t_rand, target, td, eps, "fp32", lindisp, white_bkgd,
                            netchunk)
    ref, ref_p = _oracle_grads(cfg, p, sa, sr, rays, train, t_rand, target, td, eps, lindisp, white_bkgd, netchunk)
    errs = {name: _rel(gr[:, sl], ref[:, sl]) for name, sl in GROUPS.items()}
    print(f"ray-grad fp32 train={train} K={K} B={B}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for name, e in errs.items():
        assert e <= 2e-3, (name, e)
    for n, v in ref_p.items():
        if v is None or n.startswith("alpha_linear") or n.startswith("alpha_std_linear"):
            continue
        assert _rel(gp[n], v) <= 2e-3 or (gp[n].double().cpu() - v.double()).norm().item() <= 1e-7, n


# largest relative L2 distance over the four column groups, pinned with margin (measured: see the test's docstring)
TC_BARS = {"tf32": 3e-2, "bf16": 1e-1}


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("train", [True, False])
def test_tensor_core_chains_vs_fp32(cf, dev, precision, train):
    """The tf32 and bf16 training chains against the fp32 check mode on the same call (512 rays, K = 32): relative L2
    distance per column group, pinned at the measured level with margin, like the bf16 render (the bf16 / fp16 handles
    need W >= 128).  Measured on one B200, train / test mode, worst group (o): tf32 9.4e-3 / 1.0e-2, bf16 3.1e-2 /
    3.3e-2; viewdir 1.9e-3 - 2.2e-3 (tf32) and 7.4e-3 - 7.5e-3 (bf16)."""
    cfg, p, sa, sr, rays, t_rand, target, td, g = _setup(32, 512, 64, True, seed=8, W=128)
    eps = (torch.randn(32, 1, generator=g), torch.randn(32, 3, generator=g))
    ref, _ = _library_grads(cf, dev, cfg, p, sa, sr, rays, train, t_rand, target, td, eps, "fp32", False, False, 65536)
    gr, _ = _library_grads(cf, dev, cfg, p, sa, sr, rays, train, t_rand, target, td, eps, precision, False, False, 65536)
    errs = {name: _rel(gr[:, sl], ref[:, sl]) for name, sl in GROUPS.items()}
    print(f"\nray-grad {precision} vs fp32 train={train}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for name, e in errs.items():
        assert e <= TC_BARS[precision], (name, e)


def _pose(rx, ry, rz, t):
    """c2w (3,4) from an axis-angle rotation (Rodrigues) and a translation."""
    w = torch.stack([rx, ry, rz])
    th = w.norm() + 1e-12
    k = w / th
    z = torch.zeros_like(th)
    Kx = torch.stack([torch.stack([z, -k[2], k[1]]), torch.stack([k[2], z, -k[0]]), torch.stack([-k[1], k[0], z])])
    R = torch.eye(3, dtype=w.dtype, device=w.device) + torch.sin(th) * Kx + (1 - torch.cos(th)) * (Kx @ Kx)
    return torch.cat([R, t[:, None]], 1)


@pytest.mark.parametrize("ndc", [False, True])
def test_pose_gradient_vs_oracle(cf, dev, ndc):
    """rays_from_pose + render_rays (test mode, fp32): d loss / d c2w against oracle get_rays / ndc_rays + autograd."""
    cfg = O.CfnConfig(K=16, **CFG)
    p = O.make_params(cfg, 4, "lively")
    sa, sr = O.make_latents(cfg, 4)
    H, W, focal = 12, 16, 14.0
    near, far = (0., 1.) if ndc else (2., 6.)
    c2w = torch.tensor([[0.98, -0.1, 0.17, 0.2], [0.12, 0.99, -0.05, -0.1], [-0.16, 0.07, 0.98, 0.8 if ndc else 0.3]])
    g = torch.Generator().manual_seed(2)
    A = torch.randn(H * W, 3, 16, generator=g)
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev).requires_grad_(False)
    c = c2w.to(dev).requires_grad_(True)
    rays = cf.rays_from_pose(H, W, focal, c, near, far, ndc)
    out = cf.render_rays(rays, net, None, 128, False, False, precision="fp32")
    ((out["rgb_map"] * A.to(dev)).sum() + 0.1 * out["depth_map"].sum()).backward()
    cr = c2w.clone().requires_grad_(True)
    ro, rd = O.get_rays(H, W, focal, cr)
    vd = rd / rd.norm(dim=-1, keepdim=True)
    if ndc:
        ro, rd = O.ndc_rays(H, W, focal, 1.0, ro, rd)
    nf = torch.ones_like(rd[..., :1])
    rr = torch.cat([ro, rd, near * nf, far * nf, vd], -1).reshape(-1, 11)
    ea, er = O.test_latents(sa, sr)
    o = O.render_rays(p, cfg, rr, ea, er, False, faithful=False)
    ((o["rgb_map"] * A).sum() + 0.1 * o["depth_map"].sum()).backward()
    e = _rel(c.grad, cr.grad)
    print(f"pose grad ndc={ndc}: rel L2 {e:.2e}")
    assert e <= 2e-3, e


def test_bitwise_repeatable_and_frozen_network(cf, dev):
    """Two identical calls give bitwise equal g_rays and g_c2w; a frozen network (no parameter needs a gradient:
    grads = NULL, no weight gradient at all) gives the same g_rays bit for bit and leaves every .grad untouched."""
    cfg, p, sa, sr, rays, t_rand, target, td, g = _setup(32, 300, 20, True, seed=5)
    eps = (torch.randn(32, 1, generator=g), torch.randn(32, 3, generator=g))
    a, _ = _library_grads(cf, dev, cfg, p, sa, sr, rays, True, t_rand, target, td, eps, "tf32", False, False, 65536)
    b, _ = _library_grads(cf, dev, cfg, p, sa, sr, rays, True, t_rand, target, td, eps, "tf32", False, False, 65536)
    c, gp = _library_grads(cf, dev, cfg, p, sa, sr, rays, True, t_rand, target, td, eps, "tf32", False, False, 65536,
                           params_grad=False)
    assert torch.equal(a, b) and torch.equal(a, c)
    assert all(v is None for v in gp.values())
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev).requires_grad_(False)
    grads = []
    for _ in range(2):
        pose = torch.tensor([[1., 0, 0, 0.1], [0, 1, 0, 0], [0, 0, 1, 0.2]], device=dev, requires_grad=True)
        out = cf.render_rays(cf.rays_from_pose(16, 16, 15.0, pose, 2., 6.), net, None, 128, False, False)
        out["rgb_map"].mean().backward()
        grads.append(pose.grad.clone())
    assert torch.equal(grads[0], grads[1])


def test_parameter_gradients_unchanged_by_ray_gradients(cf, dev):
    """Deterministic mode: the parameter gradients are bitwise equal with and without ray_batch.requires_grad."""
    cfg, p, sa, sr, rays, t_rand, target, td, g = _setup(16, 256, 0, True, seed=6)
    ea, er = torch.randn(16, 1, generator=g), torch.randn(16, 3, generator=g)
    res = []
    for need in (False, True):
        net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev)
        cf.engine_for(net, dev, "tf32").set_deterministic(True)
        r = rays.to(dev).requires_grad_(need)
        out = cf.render_rays(r, net, None, 128, True, False, perturb=1., t_rand=t_rand.to(dev), eps_alpha=ea.to(dev),
                             eps_rgb=er.to(dev), precision="tf32")
        cf.trainer_loss(out, target.to(dev), 16)["loss"].backward()
        res.append({n: q.grad.clone() for n, q in net.named_parameters() if q.grad is not None})
    assert res[0].keys() == res[1].keys()
    for n in res[0]:
        assert torch.equal(res[0][n], res[1][n]), n


def test_value_errors(cf, dev):
    cfg = O.CfnConfig(K=8, **dict(CFG, W=128))
    p = O.make_params(cfg, 0, "lively")
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, p).to(dev)
    rays = O.synthetic_rays(8).to(dev).requires_grad_(True)
    with pytest.raises(ValueError):
        cf.render_rays(rays, net, None, 64, True, False, N_importance=64, network_fine=net, perturb=1.)
    with pytest.raises(ValueError):
        cf.render_rays(rays, net, None, 128, False, False, want_kstats=True)
    with torch.no_grad():      # no graph wanted: the ordinary test-mode render, kstats included
        assert "kstats" in cf.render_rays(rays, net, None, 128, False, False, want_kstats=True)


def test_pose_refinement_end_to_end(cf, dev):
    """Render a 32 x 32 target from a pose, perturb the pose by ~3 degrees and ~3 % of the scene depth range, and run
    30 Adam steps on (axis-angle, translation) with the network frozen (tf32 training chain).  Measured on one B200
    (1000 W power limit): the pose error falls from 0.1905 to 0.1105 (ratio 0.580; every kernel on this path is
    bitwise repeatable); the bar is 0.75 of the start."""
    cfg = O.CfnConfig(K=16, **CFG)
    p = O.make_params(cfg, 1, "lively")
    sa, sr = O.make_latents(cfg, 1)
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev).requires_grad_(False)
    H = W = 32
    focal = 30.0
    w_true = torch.tensor([0.05, -0.1, 0.02], device=dev)
    t_true = torch.tensor([0.1, -0.05, 0.3], device=dev)
    with torch.no_grad():
        target = cf.render_rays(cf.rays_from_pose(H, W, focal, _pose(*w_true, t_true), 2., 6.), net, None, 128, False,
                                False, precision="tf32")["rgb_map"].mean(-1)
    w = (w_true + torch.tensor([0.03, 0.03, -0.03], device=dev)).requires_grad_(True)     # ~3 degrees
    t = (t_true + torch.tensor([0.08, -0.08, 0.08], device=dev)).requires_grad_(True)     # ~3 % of far - near = 4
    err0 = ((w - w_true).norm() + (t - t_true).norm()).item()
    opt = torch.optim.Adam([w, t], lr=4e-3)
    for _ in range(30):
        opt.zero_grad()
        rays = cf.rays_from_pose(H, W, focal, _pose(*w, t), 2., 6.)
        rgb = cf.render_rays(rays, net, None, 128, False, False, precision="tf32")["rgb_map"].mean(-1)
        ((rgb - target) ** 2).mean().backward()
        opt.step()
    err1 = ((w - w_true).norm() + (t - t_true).norm()).item()
    print(f"\npose refinement: error {err0:.4f} -> {err1:.4f} (ratio {err1 / err0:.3f})")
    assert err1 <= 0.75 * err0, (err0, err1)
