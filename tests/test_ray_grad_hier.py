"""Ray and pose gradients through the coarse+fine render (render_rays(..., detach_z_samples=True)) on the GPU.

fp32 check mode against the autograd of the hierarchical reference (tests/hier_oracle.py, fed the library's z_samples),
the merge permutation, the pose gradient through an NDC coarse+fine render, the tensor-core chains against fp32,
bitwise repeatability and frozen networks, the one-warp flow/compositing backward with ray gradients, and an end-to-end
coarse+fine pose refinement."""
import pytest
import torch

import hier_oracle as H
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


def _setup(K, B, Nc, Nf, n_depth, perturb, seed=3, W=64, near=2.0, far=6.0):
    cfg = O.CfnConfig(K=K, **dict(CFG, W=W))
    pc, pf = O.make_params(cfg, seed, "lively"), O.make_params(cfg, seed + 1, "lively")
    sa, sr = O.make_latents(cfg, seed)
    g = torch.Generator().manual_seed(seed + 10)
    rays = O.synthetic_rays(B, seed + 1, near=near, far=far)
    rays[:, 3:6] *= (0.7 + 0.6 * torch.rand(B, 1, generator=g))      # |d| != 1
    t_rand = torch.rand(B, Nc, generator=g) if perturb else None
    u = torch.rand(B, Nf, generator=g) if perturb else None
    target = torch.rand(B - n_depth, 3, generator=g)
    td = (3.0 + torch.rand(n_depth, generator=g)) if n_depth else None
    eps = (torch.randn(K, 1, generator=g), torch.randn(K, 3, generator=g))
    return cfg, pc, pf, sa, sr, rays, t_rand, u, target, td, eps


def _both_losses(cf, out, target, td, K, train):
    """trainer_loss on the fine maps + on the coarse maps (rgb0 / depth0 / loss_entropy0)."""
    dev = out["rgb_map"].device
    beta = 0.01 if train else 0.0
    zero = torch.zeros(1, 1, 1, device=dev)
    fine = dict(out, loss_entropy=out["loss_entropy"] if train else zero)
    coarse = dict(rgb_map=out["rgb0"], depth_map=out["depth0"], loss_entropy=out["loss_entropy0"] if train else zero)
    kw = dict(target_depth=td.to(dev) if td is not None else None, depth_lambda=0.5)
    return (cf.trainer_loss(fine, target.to(dev), K, beta, **kw)["loss"]
            + cf.trainer_loss(coarse, target.to(dev), K, beta, **kw)["loss"])


def _library(cf, dev, cfg, pc, pf, sa, sr, rays, train, Nc, Nf, t_rand, u, target, td, eps, precision, lindisp=False,
             white_bkgd=False, params_grad=True):
    net_c = cf.NeRFFlowsParams.from_oracle_params(cfg, pc, sa, sr).to(dev).requires_grad_(params_grad)
    net_f = cf.NeRFFlowsParams.from_oracle_params(cfg, pf, sa, sr).to(dev).requires_grad_(params_grad)
    r = rays.to(dev).requires_grad_(True)
    kw = dict(eps_alpha=eps[0].to(dev), eps_rgb=eps[1].to(dev)) if train else {}
    out = cf.render_rays(r, net_c, None, Nc, train, False, K_samples=cfg.K, perturb=1. if t_rand is not None else 0.,
                         N_importance=Nf, network_fine=net_f, t_rand=t_rand.to(dev) if t_rand is not None else None,
                         u=u.to(dev) if u is not None else None, precision=precision, lindisp=lindisp,
                         white_bkgd=white_bkgd, detach_z_samples=True, **kw)
    _both_losses(cf, out, target, td, cfg.K, train).backward()
    torch.cuda.synchronize()
    grads = {tag: {n: q.grad for n, q in net.named_parameters()} for tag, net in (("coarse", net_c), ("fine", net_f))}
    return r.grad.detach().cpu(), grads, out["z_samples"].cpu()


def _oracle_loss(out, target, td, K, train, ent_key, rgb_key, depth_key):
    nb = target.shape[0]
    ent = out[ent_key] if train else 0.0
    loss = O.kde_nll_loss(out[rgb_key][:nb], target, ent, K, 0.01 if train else 0.0)["loss"]
    if td is not None:
        loss = loss + 0.5 * torch.mean((out[depth_key].mean(-1)[nb:] - td) ** 2)
    return loss


def _oracle(cfg, pc, pf, sa, sr, rays, train, Nc, Nf, t_rand, z_s, target, td, eps, lindisp=False, white_bkgd=False):
    prc = {k: v.clone().requires_grad_(True) for k, v in pc.items()}
    prf = {k: v.clone().requires_grad_(True) for k, v in pf.items()}
    r = rays.clone().requires_grad_(True)
    ea, er = eps if train else O.test_latents(sa, sr)
    out = H.render_rays_hier(prc, prf, cfg, r, ea, er, train, Nc, Nf, t_rand=t_rand, lindisp=lindisp,
                             white_bkgd=white_bkgd, z_samples=z_s)
    loss = (_oracle_loss(out, target, td, cfg.K, train, "loss_entropy", "rgb_map", "depth_map")
            + _oracle_loss(out, target, td, cfg.K, train, "loss_entropy0", "rgb0", "depth0"))
    loss.backward()
    return r.grad, {"coarse": {k: v.grad for k, v in prc.items()}, "fine": {k: v.grad for k, v in prf.items()}}


# (train, Nc, Nf, B, depth rays, perturb, lindisp, white_bkgd): Nc + Nf = 66 is not a multiple of 16, so the fine pass
# takes the one-warp flow/compositing backward
CASES = [
    (True, 64, 128, 37, 7, True, False, False),
    (True, 64, 64, 700, 100, True, True, True),
    (True, 36, 30, 37, 0, False, False, True),
    (True, 64, 128, 1, 0, False, True, False),
    (False, 64, 128, 700, 100, False, False, False),
    (False, 64, 64, 37, 7, True, False, True),
    (False, 36, 30, 1, 0, True, True, False),
    (False, 36, 30, 700, 50, True, False, False),
]


@pytest.mark.parametrize("train,Nc,Nf,B,n_depth,perturb,lindisp,white_bkgd", CASES)
def test_fp32_hier_ray_gradient_vs_oracle_autograd(cf, dev, train, Nc, Nf, B, n_depth, perturb, lindisp, white_bkgd):
    """ray_batch.grad after a coarse+fine render_rays + both trainer losses, fp32 check mode, against the reference's
    autograd fed the library's z_samples: relative L2 per column group within 2e-3; in train mode both networks'
    parameter gradients within the 2e-2 bar of the coarse+fine training test."""
    cfg, pc, pf, sa, sr, rays, t_rand, u, target, td, eps = _setup(16, B, Nc, Nf, n_depth, perturb)
    gr, gp, z_s = _library(cf, dev, cfg, pc, pf, sa, sr, rays, train, Nc, Nf, t_rand, u, target, td, eps, "fp32",
                           lindisp, white_bkgd)
    ref, ref_p = _oracle(cfg, pc, pf, sa, sr, rays, train, Nc, Nf, t_rand, z_s, target, td, eps, lindisp, white_bkgd)
    errs = {name: _rel(gr[:, sl], ref[:, sl]) for name, sl in GROUPS.items()}
    print(f"hier ray-grad fp32 train={train} Nc={Nc} Nf={Nf} B={B}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for name, e in errs.items():
        assert e <= 2e-3, (name, e)
    if train:
        for tag in ("coarse", "fine"):
            for n, v in ref_p[tag].items():
                if v is None or v.norm() == 0 or n.startswith("alpha_linear") or n.startswith("alpha_std_linear"):
                    continue
                assert gp[tag][n] is not None, (tag, n)
                assert _rel(gp[tag][n], v) <= 2e-2, (tag, n, _rel(gp[tag][n], v))


@pytest.mark.parametrize("Na,Nb", [(64, 128), (36, 30), (1, 5), (128, 0)])
def test_merge_permutation(cf, dev, Na, Nb):
    """merge_sorted(..., return_src=True): the values are bitwise those of the values-only merge, src reproduces them
    and equals torch.sort(stable=True).indices, constructed ties included."""
    g = torch.Generator().manual_seed(Na + Nb)
    B = 300
    a = torch.sort(torch.rand(B, Na, generator=g), -1).values
    b = torch.rand(B, Nb, generator=g)
    if Nb >= 8 and Na >= 8:
        b[:, :4] = a[:, :4]           # ties between the two inputs
        b[:, 4:6] = b[:, 6:8]         # ties inside b
        a[:, 1] = a[:, 0]             # ties inside a
    out, src = cf.merge_sorted(a.to(dev), b.to(dev), return_src=True)
    vals = cf.merge_sorted(a.to(dev), b.to(dev))
    assert src.dtype == torch.int32
    assert torch.equal(out, vals)
    cat = torch.cat([a, b], -1)
    assert torch.equal(torch.gather(cat, -1, src.long().cpu()), out.cpu())
    assert torch.equal(src.long().cpu(), torch.sort(cat, dim=-1, stable=True).indices)


def _pose(rx, ry, rz, t):
    """c2w (3,4) from an axis-angle rotation (Rodrigues) and a translation."""
    w = torch.stack([rx, ry, rz])
    th = w.norm() + 1e-12
    k = w / th
    z = torch.zeros_like(th)
    Kx = torch.stack([torch.stack([z, -k[2], k[1]]), torch.stack([k[2], z, -k[0]]), torch.stack([-k[1], k[0], z])])
    R = torch.eye(3, dtype=w.dtype, device=w.device) + torch.sin(th) * Kx + (1 - torch.cos(th)) * (Kx @ Kx)
    return torch.cat([R, t[:, None]], 1)


def test_pose_gradient_through_ndc_coarse_fine_vs_oracle(cf, dev):
    """rays_from_pose (NDC) + coarse+fine render_rays (test mode, fp32, frozen networks): d loss / d c2w against oracle
    get_rays / ndc_rays + the hierarchical reference's autograd, fed the library's z_samples."""
    cfg = O.CfnConfig(K=16, **CFG)
    pc, pf = O.make_params(cfg, 4, "lively"), O.make_params(cfg, 5, "lively")
    sa, sr = O.make_latents(cfg, 4)
    H_, W_, focal, Nc, Nf = 12, 16, 14.0, 64, 64
    c2w = torch.tensor([[0.98, -0.1, 0.17, 0.2], [0.12, 0.99, -0.05, -0.1], [-0.16, 0.07, 0.98, 0.8]])
    g = torch.Generator().manual_seed(2)
    A = torch.randn(H_ * W_, 3, 16, generator=g)
    net_c = cf.NeRFFlowsParams.from_oracle_params(cfg, pc, sa, sr).to(dev).requires_grad_(False)
    net_f = cf.NeRFFlowsParams.from_oracle_params(cfg, pf, sa, sr).to(dev).requires_grad_(False)
    c = c2w.to(dev).requires_grad_(True)
    rays = cf.rays_from_pose(H_, W_, focal, c, 0., 1., True)
    out = cf.render_rays(rays, net_c, None, Nc, False, False, N_importance=Nf, network_fine=net_f, precision="fp32",
                         detach_z_samples=True)
    ((out["rgb_map"] * A.to(dev)).sum() + 0.1 * out["depth_map"].sum() + 0.5 * (out["rgb0"] * A.to(dev)).sum()).backward()
    cr = c2w.clone().requires_grad_(True)
    ro, rd = O.get_rays(H_, W_, focal, cr)
    vd = rd / rd.norm(dim=-1, keepdim=True)
    ro, rd = O.ndc_rays(H_, W_, focal, 1.0, ro, rd)
    nf = torch.ones_like(rd[..., :1])
    rr = torch.cat([ro, rd, 0. * nf, nf, vd], -1).reshape(-1, 11)
    ea, er = O.test_latents(sa, sr)
    o = H.render_rays_hier(pc, pf, cfg, rr, ea, er, False, Nc, Nf, z_samples=out["z_samples"].cpu())
    ((o["rgb_map"] * A).sum() + 0.1 * o["depth_map"].sum() + 0.5 * (o["rgb0"] * A).sum()).backward()
    e = _rel(c.grad, cr.grad)
    print(f"hier pose grad ndc: rel L2 {e:.2e}")
    assert e <= 2e-3, e


# largest relative L2 distance over the four column groups, pinned with margin (measured: see the test's docstring)
TC_BARS = {"tf32": 5e-2, "bf16": 1.5e-1}


@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("train", [True, False])
def test_hier_tensor_core_chains_vs_fp32(cf, dev, precision, train):
    """The tf32 and bf16 chains against the fp32 check mode on the same coarse+fine call (512 rays, 64 + 128 samples,
    K = 32, W = 128), relative L2 per column group.  Each chain resamples from its own coarse weights, so the fine grids
    differ slightly too, and the distances are about twice the single-network ones.  Measured on one B200 (1000 W power
    limit), train / test mode, worst group (o): tf32 2.1e-2 / 2.0e-2, bf16 6.5e-2 / 7.2e-2; viewdir 2.4e-3 - 2.8e-3
    (tf32) and 7.4e-3 - 7.6e-3 (bf16)."""
    cfg, pc, pf, sa, sr, rays, t_rand, u, target, td, eps = _setup(32, 512, 64, 128, 64, True, seed=8, W=128)
    args = (cfg, pc, pf, sa, sr, rays, train, 64, 128, t_rand, u, target, td, eps)
    ref, _, _ = _library(cf, dev, *args, "fp32")
    gr, _, _ = _library(cf, dev, *args, precision)
    errs = {name: _rel(gr[:, sl], ref[:, sl]) for name, sl in GROUPS.items()}
    print(f"\nhier ray-grad {precision} vs fp32 train={train}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for name, e in errs.items():
        assert e <= TC_BARS[precision], (name, e)


def test_hier_bitwise_repeatable_and_frozen_networks(cf, dev):
    """Two identical coarse+fine calls give bitwise equal g_rays and g_c2w; a frozen pair of networks gives the same
    g_rays bit for bit and leaves every .grad untouched."""
    cfg, pc, pf, sa, sr, rays, t_rand, u, target, td, eps = _setup(32, 300, 64, 128, 20, True, seed=5)
    args = (cfg, pc, pf, sa, sr, rays, True, 64, 128, t_rand, u, target, td, eps, "tf32")
    a, _, _ = _library(cf, dev, *args)
    b, _, _ = _library(cf, dev, *args)
    c, gp, _ = _library(cf, dev, *args, params_grad=False)
    assert torch.equal(a, b) and torch.equal(a, c)
    assert all(v is None for grads in gp.values() for v in grads.values())
    net_c = cf.NeRFFlowsParams.from_oracle_params(cfg, pc, sa, sr).to(dev).requires_grad_(False)
    net_f = cf.NeRFFlowsParams.from_oracle_params(cfg, pf, sa, sr).to(dev).requires_grad_(False)
    grads = []
    for _ in range(2):
        pose = torch.tensor([[1., 0, 0, 0.1], [0, 1, 0, 0], [0, 0, 1, 0.3]], device=dev, requires_grad=True)
        out = cf.render_rays(cf.rays_from_pose(16, 16, 15.0, pose, 0., 1., True), net_c, None, 64, False, False,
                             N_importance=128, network_fine=net_f, detach_z_samples=True)
        (out["rgb_map"].mean() + out["rgb0"].mean()).backward()
        grads.append(pose.grad.clone())
    assert torch.equal(grads[0], grads[1])
    assert all(q.grad is None for net in (net_c, net_f) for q in net.parameters())


def _single_oracle(p, cfg, rays, ea, er, N):
    """O.render_rays for a linspace(0, 1, N) schedule (O.render_rays has the reference's 128 samples)."""
    z = O.z_from_t(torch.linspace(0., 1., steps=N), rays[:, 6:7], rays[:, 7:8], False)
    pts = rays[:, None, 0:3] + rays[:, None, 3:6] * z[..., None]
    raw, _ = O.run_network(p, cfg, pts, rays[:, -3:], ea, er, False, faithful=False)
    return O.raw2outputs(raw, z, rays[:, 3:6])


def test_one_warp_backward_with_ray_gradients(cf, dev):
    """The one-warp flow/compositing backward (16 384 rays, or N not a multiple of 16) with ray gradients, single
    network, fp32 check mode, test mode: the first 700 rays of a 16 384-ray batch (sum loss) get the gradient they get
    when rendered alone (segmented backward), within fp32 summation-order noise; with N_samples = 100 the gradient
    matches the reference's autograd at 2e-3."""
    cfg = O.CfnConfig(K=16, **CFG)
    p = O.make_params(cfg, 7, "lively")
    sa, sr = O.make_latents(cfg, 7)
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev).requires_grad_(False)
    rays = O.synthetic_rays(16384, 9, near=2.0, far=6.0)
    A = torch.randn(16384, 3, 16, generator=torch.Generator().manual_seed(3)).to(dev)
    res = []
    for n in (16384, 700):
        r = rays[:n].to(dev).requires_grad_(True)
        out = cf.render_rays(r, net, None, 128, False, False, precision="fp32")
        ((out["rgb_map"] * A[:n]).sum() + 0.1 * out["depth_map"].sum()).backward()
        res.append(r.grad[:700].cpu())
    errs = {name: _rel(res[0][:, sl], res[1][:, sl]) for name, sl in GROUPS.items()}
    print("one-warp vs segmented: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for name, e in errs.items():
        assert e <= 1e-5, (name, e)
    r = rays[:300].to(dev).requires_grad_(True)
    out = cf.render_rays(r, net, None, 100, False, False, precision="fp32")
    ((out["rgb_map"] * A[:300]).sum() + 0.1 * out["depth_map"].sum()).backward()
    rr = rays[:300].clone().requires_grad_(True)
    ea, er = O.test_latents(sa, sr)
    rgb, _, _, depth = _single_oracle(p, cfg, rr, ea, er, 100)
    ((rgb * A[:300].cpu()).sum() + 0.1 * depth.sum()).backward()
    errs = {name: _rel(r.grad[:, sl], rr.grad[:, sl]) for name, sl in GROUPS.items()}
    print("N = 100 vs oracle: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for name, e in errs.items():
        assert e <= 2e-3, (name, e)


def test_coarse_fine_pose_refinement_end_to_end(cf, dev):
    """Render a 32 x 32 NDC target with a coarse+fine pair (64 + 64 samples) from a pose, perturb the pose by ~3 degrees
    and a translation of ~0.14, and run 30 Adam steps on (axis-angle, translation) with both networks frozen (tf32
    training chain, detach_z_samples=True).  Measured on one B200 (1000 W power limit): the pose error falls from 0.1905
    to 0.1258 (ratio 0.660); the bar is 0.75 of the start."""
    cfg = O.CfnConfig(K=16, **CFG)
    pc, pf = O.make_params(cfg, 1, "lively"), O.make_params(cfg, 2, "lively")
    sa, sr = O.make_latents(cfg, 1)
    net_c = cf.NeRFFlowsParams.from_oracle_params(cfg, pc, sa, sr).to(dev).requires_grad_(False)
    net_f = cf.NeRFFlowsParams.from_oracle_params(cfg, pf, sa, sr).to(dev).requires_grad_(False)
    H_ = W_ = 32
    focal = 30.0
    kw = dict(N_importance=64, network_fine=net_f, precision="tf32", detach_z_samples=True)
    w_true = torch.tensor([0.05, -0.1, 0.02], device=dev)
    t_true = torch.tensor([0.1, -0.05, 0.3], device=dev)
    with torch.no_grad():
        target = cf.render_rays(cf.rays_from_pose(H_, W_, focal, _pose(*w_true, t_true), 0., 1., True), net_c, None, 64,
                                False, False, **kw)["rgb_map"].mean(-1)
    w = (w_true + torch.tensor([0.03, 0.03, -0.03], device=dev)).requires_grad_(True)     # ~3 degrees
    t = (t_true + torch.tensor([0.08, -0.08, 0.08], device=dev)).requires_grad_(True)
    err0 = ((w - w_true).norm() + (t - t_true).norm()).item()
    opt = torch.optim.Adam([w, t], lr=4e-3)
    for _ in range(30):
        opt.zero_grad()
        rays = cf.rays_from_pose(H_, W_, focal, _pose(*w, t), 0., 1., True)
        rgb = cf.render_rays(rays, net_c, None, 64, False, False, **kw)["rgb_map"].mean(-1)
        ((rgb - target) ** 2).mean().backward()
        opt.step()
    err1 = ((w - w_true).norm() + (t - t_true).norm()).item()
    print(f"\ncoarse+fine pose refinement: error {err0:.4f} -> {err1:.4f} (ratio {err1 / err0:.3f})")
    assert err1 <= 0.75 * err0, (err0, err1)
