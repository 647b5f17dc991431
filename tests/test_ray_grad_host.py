"""F7 on the host: the oracle's autograd with respect to the ray record is a valid reference (central finite differences
in float64), it matches the unmodified reference's autograd where that is available, and the new C-ABI entry points
reject null pointers and bad shapes before any CUDA call."""
import ctypes as C

import pytest
import torch

from oracle import cfnerf_oracle as O
from oracle import refload

TINY = O.CfnConfig(D=4, W=16, L_pos=3, L_dir=2, h_alpha=8, h_rgb=8, F=2, K=4)
GROUPS = {"o": slice(0, 3), "d": slice(3, 6), "near/far": slice(6, 8), "viewdir": slice(8, 11)}


def _objective(p, cfg, rays, ea, er, train, t_rand, lindisp, white_bkgd, A, Bm):
    out = O.render_rays(p, cfg, rays, ea, er, train, t_rand=t_rand, lindisp=lindisp, white_bkgd=white_bkgd,
                        faithful=False)
    L = (out["rgb_map"] * A).sum() + (out["depth_map"] * Bm).sum()
    if train:
        L = L + 0.3 * out["loss_entropy"]
    return L


@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("lindisp,white_bkgd,perturb", [(False, False, False), (True, True, True), (False, True, True),
                                                         (True, False, False)])
def test_oracle_ray_gradient_matches_finite_differences(train, lindisp, white_bkgd, perturb):
    cfg = TINY
    p = O._cast(O.make_params(cfg, 3, "lively"), torch.float64)
    g = torch.Generator().manual_seed(11)
    B = 2
    rays = O.synthetic_rays(B, 5, near=2.0, far=6.0).double()
    rays[:, 3:6] *= torch.tensor([1.3, 0.8])[:, None].double()      # |d| != 1: exercises the |d| in the sample distances
    ea, er = torch.randn(cfg.K, 1, generator=g).double(), torch.randn(cfg.K, 3, generator=g).double()
    t_rand = torch.rand(B, 128, generator=g).double() if perturb else None
    A, Bm = torch.randn(B, 3, cfg.K, generator=g).double(), 0.1 * torch.randn(B, cfg.K, generator=g).double()
    args = (ea, er, train, t_rand, lindisp, white_bkgd, A, Bm)
    r = rays.clone().requires_grad_(True)
    _objective(p, cfg, r, *args).backward()
    fd = torch.zeros_like(rays)
    h = 1e-6
    for b in range(B):
        for j in range(11):
            rp, rm = rays.clone(), rays.clone()
            rp[b, j] += h
            rm[b, j] -= h
            with torch.no_grad():
                fd[b, j] = (_objective(p, cfg, rp, *args) - _objective(p, cfg, rm, *args)) / (2 * h)
    for name, sl in GROUPS.items():
        err = (r.grad[:, sl] - fd[:, sl]).norm().item()
        assert err <= 1e-6 * max(fd[:, sl].norm().item(), 1e-3), (name, err, fd[:, sl].norm().item())


@pytest.mark.reference
@pytest.mark.skipif(not refload.reference_available(), reason="reference tree not present")
@pytest.mark.parametrize("train", [False, True])
def test_oracle_ray_gradient_matches_the_reference_autograd(train):
    """The reference's render_rays is one autograd graph from ray_batch: its gradient for all 11 columns equals the
    oracle's (perturb on in train mode, with the same stratified draws)."""
    cfg = O.CfnConfig(D=4, W=64, K=8, h_alpha=16, h_rgb=16)
    p = O.make_params(cfg, 2, "lively")
    sa, sr = O.make_latents(cfg, 2)
    main, model, nq = refload.build_reference_model(cfg, p, sa, sr)
    B = 6
    rays = O.synthetic_rays(B, 9)
    A = torch.randn(B, 3, cfg.K, generator=torch.Generator().manual_seed(1))
    r1 = rays.clone().requires_grad_(True)
    torch.manual_seed(5)
    ref = main.render_rays(r1, model, nq, 128, train, False, K_samples=cfg.K, perturb=1.0 if train else 0.0,
                           raw_noise_std=0.0)
    ((ref["rgb_map"] * A).sum() + ref["depth_map"].sum()).backward()
    torch.manual_seed(5)
    t_rand = torch.rand(B, 128) if train else None
    if train:
        ea, er = torch.empty(cfg.K, 1).normal_(), torch.empty(cfg.K, 3).normal_()
    else:
        ea, er = O.test_latents(sa, sr)
    r2 = rays.clone().requires_grad_(True)
    mine = O.render_rays(p, cfg, r2, ea, er, train, t_rand=t_rand)
    ((mine["rgb_map"] * A).sum() + mine["depth_map"].sum()).backward()
    for name, sl in GROUPS.items():
        err = (r1.grad[:, sl] - r2.grad[:, sl]).norm().item()
        assert err <= 1e-5 * max(r1.grad[:, sl].norm().item(), 1e-6), (name, err)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from cfnerf_b200 import _lib
    return _lib.load()


def test_ray_gradient_entry_points_check_arguments_before_cuda(lib):
    P = C.c_void_p(4096)      # never dereferenced: every call below must fail in its argument check
    assert lib.cfn_input_grad_width(None) == 0
    # cfn_flow_composite_bwd_rays: bad shape, then null handle / pointers
    fb = lib.cfn_flow_composite_bwd_rays
    assert fb(None, P, P, P, 11, P, P, 0, -1, 128, 0, P, None, P, P, None, 1, P, P, P, P, None) == -1
    assert b"bad shape" in lib.cfn_last_error()
    assert fb(None, P, P, P, 11, P, P, 0, 4, 1, 0, P, None, P, P, None, 1, P, P, P, P, None) == -1
    assert fb(None, P, P, P, 11, P, P, 0, 4, 128, 0, P, None, P, P, None, 1, P, P, P, P, None) == -1
    assert b"null argument" in lib.cfn_last_error()
    assert fb(P, P, P, P, 11, P, P, 0, 4, 128, 0, P, None, P, P, None, 1, P, P, None, P, None) == -1
    # cfn_network_bwd_inputs
    nb = lib.cfn_network_bwd_inputs
    assert nb(P, P, -3, 128, P, 1 << 20, None, 0, P, None) == -1
    assert b"bad shape" in lib.cfn_last_error()
    assert nb(P, P, 4, 0, P, 1 << 20, None, 0, P, None) == -1
    assert nb(None, P, 4, 128, P, 1 << 20, None, 0, P, None) == -1
    assert nb(P, P, 4, 128, P, 1 << 20, None, 0, None, None) == -1
    assert b"null argument" in lib.cfn_last_error()
    # cfn_ray_grad_f32
    rg = lib.cfn_ray_grad_f32
    assert rg(P, P, P, P, None, 0, P, P, P, -1, 128, P, None) == -1
    assert rg(P, P, P, P, None, 0, P, P, P, 4, 0, P, None) == -1
    assert b"bad shape" in lib.cfn_last_error()
    assert rg(None, P, P, P, None, 0, P, P, P, 4, 128, P, None) == -1
    assert b"null handle" in lib.cfn_last_error()
    # cfn_rays_from_pose_bwd_f32
    pb = lib.cfn_rays_from_pose_bwd_f32
    assert pb(0, 16, 20.0, P, 0, 1.0, P, P, P, None) == -1
    assert pb(12, 16, -1.0, P, 0, 1.0, P, P, P, None) == -1
    assert b"bad image size" in lib.cfn_last_error()
    for k in range(4):
        args = [P, P, P, P]
        args[k] = None
        assert pb(12, 16, 20.0, args[0], 0, 1.0, args[1], args[2], args[3], None) == -1
        assert b"null argument" in lib.cfn_last_error()


def test_ray_gradient_errors_are_raised_before_any_device_work():
    """Coarse+fine and want_kstats with a ray gradient are refused as ValueError (the checks precede the engine)."""
    import cfnerf_b200 as cf
    net = cf.NeRFFlowsParams(netwidth=64, K_samples=4)
    rays = O.synthetic_rays(4).requires_grad_(True)
    with pytest.raises(ValueError, match="single-network"):
        cf.render_rays(rays, net, None, 64, False, False, N_importance=32, network_fine=net)
    with pytest.raises(ValueError, match="want_kstats"):
        cf.render_rays(rays, net, None, 128, False, False, want_kstats=True)
