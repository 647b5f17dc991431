"""Pin the oracle restatement to the UNMODIFIED reference executed live.

The reference is not part of this repository: these tests run where oracle/refload.py finds a copy of it and skip
elsewhere.  Without it, the committed fixtures under tests/golden/ (which the reference generated) still pin
render_rays in test and train mode, raw2outputs, the network and the trainer body; nothing stored replaces the live
checks of get_rays / ndc_rays and of the D=7 model without a skip connection.
"""
import pytest
import torch

from oracle import cfnerf_oracle as O
from oracle import refload

pytestmark = pytest.mark.skipif(not refload.reference_available(), reason="reference tree not present")


@pytest.mark.parametrize("variant,seed", [("default", 0), ("lively", 4)])
def test_render_rays_test_mode_live(variant, seed):
    cfg = O.CfnConfig()
    p = O.make_params(cfg, seed, variant)
    sa, sr = O.make_latents(cfg, seed)
    main, model, nq = refload.build_reference_model(cfg, p, sa, sr)
    rays = O.synthetic_rays(12, seed + 1)
    with torch.no_grad():
        ref = main.render_rays(rays, model, nq, 128, False, False, K_samples=cfg.K, perturb=0.0, raw_noise_std=0.0)
        ea, er = O.test_latents(sa, sr)
        mine = O.render_rays(p, cfg, rays, ea, er, False)
    for k in ("rgb_map", "disp_map", "depth_map"):
        assert (ref[k] - mine[k]).abs().max().item() <= 2e-6, k


def test_render_rays_train_mode_live_rng_order():
    cfg = O.CfnConfig(W=256, K=64, h_alpha=32)
    p = O.make_params(cfg, 7, "lively")
    sa, sr = O.make_latents(cfg, 7)
    main, model, nq = refload.build_reference_model(cfg, p, sa, sr)
    rays = O.synthetic_rays(8, 3)
    torch.manual_seed(123)
    ref = main.render_rays(rays, model, nq, 128, True, False, K_samples=cfg.K, perturb=1.0, raw_noise_std=1.0)
    torch.manual_seed(123)
    t_rand = torch.rand(8, 128)
    ea = torch.empty(cfg.K, 1).normal_()
    er = torch.empty(cfg.K, 3).normal_()
    mine = O.render_rays(p, cfg, rays, ea, er, True, t_rand=t_rand)
    for k in ("rgb_map", "disp_map", "depth_map", "raw"):
        assert (ref[k] - mine[k]).abs().max().item() <= 2e-6, k
    assert abs(ref["loss_entropy"].mean().item() - mine["loss_entropy"].item()) <= 1e-6
    assert ref["loss_entropy"].shape == (8 * 128, cfg.K, 1)  # the broadcast scalar (models:291)


def test_get_rays_and_ndc_live():
    main, _ = refload.load_reference()
    c2w = torch.eye(4)[:3]
    o_ref, d_ref = main.get_rays(12, 16, 20.0, c2w)
    o, d = O.get_rays(12, 16, 20.0, c2w)
    assert torch.equal(o_ref, o) and torch.equal(d_ref, d)
    o2r, d2r = main.ndc_rays(12, 16, 20.0, 1.0, o_ref + torch.tensor([0.0, 0.0, 0.5]), d_ref)
    o2, d2 = O.ndc_rays(12, 16, 20.0, 1.0, o + torch.tensor([0.0, 0.0, 0.5]), d)
    assert torch.equal(o2r, o2) and torch.equal(d2r, d2)


def test_odd_depth_has_no_skip_connection_live():
    """skips=[netdepth/2] uses true division (main:327): D=7 gives [3.5] and the model has no skip layer."""
    cfg = O.CfnConfig(D=7, W=64, K=8, h_alpha=16, h_rgb=16)
    assert cfg.skip == -1
    p = O.make_params(cfg, 0, "lively")
    sa, sr = O.make_latents(cfg, 0)
    main, model, nq = refload.build_reference_model(cfg, p, sa, sr)
    assert all(l.in_features == (cfg.in_pos if i == 0 else cfg.W) for i, l in enumerate(model.pts_linears))
    rays = O.synthetic_rays(6, 2)
    with torch.no_grad():
        ref = main.render_rays(rays, model, nq, 128, False, False, K_samples=cfg.K, perturb=0.0, raw_noise_std=0.0)
        ea, er = O.test_latents(sa, sr)
        mine = O.render_rays(p, cfg, rays, ea, er, False)
    assert (ref["rgb_map"] - mine["rgb_map"]).abs().max().item() <= 2e-6
