"""Ray gradients through the coarse+fine pass, on the host: the differentiable hierarchical reference (tests/hier_oracle.py,
resampled depths pinned) against float64 central differences; its stable-sort merge against the oracle's numpy merge;
the argument checks of cfn_merge_sorted_src_f32 / cfn_ray_grad_merged_f32; and the ValueErrors render_rays keeps
without detach_z_samples."""
import ctypes as C

import numpy as np
import pytest
import torch

import hier_oracle as H
from oracle import cfnerf_oracle as O

TINY = O.CfnConfig(D=4, W=16, L_pos=3, L_dir=2, h_alpha=8, h_rgb=8, F=2, K=4)
GROUPS = {"o": slice(0, 3), "d": slice(3, 6), "near/far": slice(6, 8), "viewdir": slice(8, 11)}
NC, NF = 16, 24


def _objective(pc, pf, rays, ea, er, train, t_rand, lindisp, white_bkgd, z_s, A, Bm):
    out = H.render_rays_hier(pc, pf, TINY, rays, ea, er, train, NC, NF, t_rand=t_rand, lindisp=lindisp,
                             white_bkgd=white_bkgd, z_samples=z_s)
    L = ((out["rgb_map"] * A).sum() + (out["depth_map"] * Bm).sum() + 0.7 * (out["rgb0"] * A).sum()
         + 0.4 * (out["depth0"] * Bm).sum())
    if train:
        L = L + 0.3 * out["loss_entropy"] + 0.2 * out["loss_entropy0"]
    return L


# (lindisp, white_bkgd, perturb, ndc): ndc = NDC-style rays, near = 0 and far = 1 (linear schedule only: lindisp needs
# near > 0)
@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("lindisp,white_bkgd,perturb,ndc", [(False, False, False, False), (True, True, True, False),
                                                             (False, True, True, True), (False, False, False, True)])
def test_hier_ray_gradient_matches_finite_differences(train, lindisp, white_bkgd, perturb, ndc):
    """With z_samples pinned, the hierarchical reference's autograd gradient for all 11 columns equals float64 central
    differences, at the bar of the single-network check (1e-6 relative per column group)."""
    pc = O._cast(O.make_params(TINY, 3, "lively"), torch.float64)
    pf = O._cast(O.make_params(TINY, 4, "lively"), torch.float64)
    g = torch.Generator().manual_seed(12)
    B = 2
    rays = (O.synthetic_rays(B, 5, near=0.0, far=1.0) if ndc else O.synthetic_rays(B, 5, near=2.0, far=6.0)).double()
    rays[:, 3:6] *= torch.tensor([1.3, 0.8])[:, None].double()
    ea, er = torch.randn(TINY.K, 1, generator=g).double(), torch.randn(TINY.K, 3, generator=g).double()
    t_rand = torch.rand(B, NC, generator=g).double() if perturb else None
    u = torch.rand(B, NF, generator=g) if perturb else None
    z_s = H.render_rays_hier(pc, pf, TINY, rays, ea, er, train, NC, NF, t_rand=t_rand, u=u, lindisp=lindisp,
                             white_bkgd=white_bkgd)["z_samples"].double()
    A, Bm = torch.randn(B, 3, TINY.K, generator=g).double(), 0.1 * torch.randn(B, TINY.K, generator=g).double()
    args = (ea, er, train, t_rand, lindisp, white_bkgd, z_s, A, Bm)
    r = rays.clone().requires_grad_(True)
    _objective(pc, pf, r, *args).backward()
    fd = torch.zeros_like(rays)
    h = 1e-7        # smaller than the single-network check's step: 40 more points per ray put more ReLU kinks near a ray
    for b in range(B):
        for j in range(11):
            rp, rm = rays.clone(), rays.clone()
            rp[b, j] += h
            rm[b, j] -= h
            with torch.no_grad():
                fd[b, j] = (_objective(pc, pf, rp, *args) - _objective(pc, pf, rm, *args)) / (2 * h)
    for name, sl in GROUPS.items():
        err = (r.grad[:, sl] - fd[:, sl]).norm().item()
        assert err <= 1e-6 * max(fd[:, sl].norm().item(), 1e-3), (name, err, fd[:, sl].norm().item())


def test_stable_sort_merge_equals_the_numpy_merge():
    """merge_sorted_graph gives bitwise the values of np.sort (O.merge_sorted), its permutation is the stable one
    (ties: the coarse depth first), and the reference's forward is bitwise O.render_rays_hier's."""
    g = torch.Generator().manual_seed(4)
    z_c = torch.sort(torch.rand(5, 40, generator=g) * 4 + 2, -1).values
    z_s = torch.rand(5, 56, generator=g) * 4 + 2
    z_s[:, :20] = z_c[:, ::2]                                # constructed ties with the coarse depths
    z_s[:, 20:24] = z_s[:, 24:28]                            # and among the resampled ones
    z_all, src = H.merge_sorted_graph(z_c, z_s)
    ref = O.merge_sorted(z_c.numpy(), z_s.numpy())
    assert np.array_equal(z_all.numpy().view(np.int32), ref.view(np.int32))
    cat = torch.cat([z_c, z_s], -1)
    assert torch.equal(torch.gather(cat, -1, src), z_all)
    assert torch.equal(src, torch.from_numpy(np.argsort(cat.numpy(), -1, kind="stable")))
    cfg = O.CfnConfig(D=4, W=32, K=4, h_alpha=8, h_rgb=8)
    pc, pf = O.make_params(cfg, 0, "lively"), O.make_params(cfg, 1, "lively")
    ea, er = O.make_latents(cfg, 0)
    rays = O.synthetic_rays(3, 2)
    t_rand, u = torch.rand(3, 64, generator=g), torch.rand(3, 32, generator=g)
    a = O.render_rays_hier(pc, pf, cfg, rays, ea, er, True, 64, 32, t_rand=t_rand, u=u)
    b = H.render_rays_hier(pc, pf, cfg, rays, ea, er, True, 64, 32, t_rand=t_rand, u=u)
    for k in ("z_vals", "z_samples", "rgb_map", "depth_map", "disp_map", "rgb0", "depth0", "loss_entropy"):
        assert torch.equal(a[k], b[k]), k


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from cfnerf_b200 import _lib
    return _lib.load()


def test_merged_grid_entry_points_check_arguments_before_cuda(lib):
    P = C.c_void_p(4096)      # never dereferenced: every call below must fail in its argument check
    ms = lib.cfn_merge_sorted_src_f32
    assert ms(P, P, P, P, -1, 4, 4, None) == -1
    assert ms(P, P, P, P, 2, -4, 4, None) == -1
    assert b"negative size" in lib.cfn_last_error()
    for k in range(4):
        args = [P, P, P, P]
        args[k] = None
        assert ms(*args, 2, 4, 4, None) == -1
        assert b"null argument" in lib.cfn_last_error()
    assert ms(P, P, P, P, 0, 4, 4, None) == 0          # nothing to do: no launch
    rg = lib.cfn_ray_grad_merged_f32
    #       h  rays z  src Nc t_vals t_rand lin g_enc g_zd g_dl B   N   g_rays
    assert rg(P, P, P, P, 64, P, None, 0, P, P, P, -1, 192, P, None) == -1
    assert rg(P, P, P, P, 64, P, None, 0, P, P, P, 4, 0, P, None) == -1
    assert b"bad shape" in lib.cfn_last_error()
    for nc in (0, -3, 193):
        assert rg(P, P, P, P, nc, P, None, 0, P, P, P, 4, 192, P, None) == -1
        assert b"out of range" in lib.cfn_last_error()
    assert rg(None, P, P, P, 64, P, None, 0, P, P, P, 4, 192, P, None) == -1
    assert b"null handle" in lib.cfn_last_error()
    for k in range(7):
        ptrs = [P] * 7      # rays, z_vals, src, t_vals, g_enc, g_zdirect, g_delta
        ptrs[k] = None
        assert rg(P, ptrs[0], ptrs[1], ptrs[2], 64, ptrs[3], None, 0, ptrs[4], ptrs[5], ptrs[6], 4, 192, P, None) == -1
        assert b"null argument" in lib.cfn_last_error()
    assert rg(P, P, P, P, 64, P, None, 0, P, P, P, 4, 192, None, None) == -1
    assert b"null argument" in lib.cfn_last_error()


def test_coarse_fine_ray_gradient_errors_without_detach_z_samples():
    """Without detach_z_samples the coarse+fine pass with a ray gradient keeps its ValueError (which names the keyword),
    and want_kstats keeps its own with the keyword too; both are raised before any device work."""
    import cfnerf_b200 as cf
    net = cf.NeRFFlowsParams(netwidth=64, K_samples=4)
    rays = O.synthetic_rays(4).requires_grad_(True)
    with pytest.raises(ValueError, match="single-network") as e:
        cf.render_rays(rays, net, None, 64, False, False, N_importance=32, network_fine=net)
    assert "detach_z_samples=True" in str(e.value)
    with pytest.raises(ValueError, match="single-network"):
        cf.render_rays(rays, net, None, 64, True, False, N_importance=32, network_fine=net, perturb=1.,
                       detach_z_samples=False)
    with pytest.raises(ValueError, match="want_kstats"):
        cf.render_rays(rays, net, None, 64, False, False, N_importance=32, network_fine=net, want_kstats=True,
                       detach_z_samples=True)
