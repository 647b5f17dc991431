"""The fused network + compositing kernel (Engine.network(..., composite=), cfn_network_fwd_composite) against
Engine.network followed by Engine.flow_composite on the same inputs: the maps must be bitwise equal.  Also the rule
by which render_rays picks the fused path."""
import ctypes as C
import types

import pytest
import torch

from oracle import cfnerf_oracle as O

CFN_EINVAL = -1


# ------------------------------------------------------------------------------------------------
# host only
# ------------------------------------------------------------------------------------------------
def _fake_engine(precision="fp16", F=4, K=32):
    return types.SimpleNamespace(precision=precision, F=F, K=K)


def test_dispatch_rule():
    from cfnerf_b200.api import FUSED_MAX_K, fused_composite
    assert fused_composite(_fake_engine("fp16"), 128, False, 0)
    assert fused_composite(_fake_engine("bf16"), 64, False, 0)
    assert fused_composite(_fake_engine("fp16"), 32, False, 0)
    assert not fused_composite(_fake_engine("fp32"), 128, False, 0)        # check mode: its own kernels
    assert not fused_composite(_fake_engine("tf32"), 128, False, 0)        # layer-by-layer chain
    assert not fused_composite(_fake_engine("fp16"), 128, True, 0)         # weights wanted (fern's coarse pass)
    assert not fused_composite(_fake_engine("fp16"), 192, False, 0)        # fern's fine pass: rays straddle tiles
    assert not fused_composite(_fake_engine("fp16", F=2), 128, False, 0)   # only the F = 4 flavour is compiled
    assert not fused_composite(_fake_engine("fp16"), 128, False, 512)      # several latent-draw groups
    assert not fused_composite(_fake_engine("fp16", K=FUSED_MAX_K + 1), 128, False, 0)


def test_cabi_rejects_bad_arguments_on_the_host():
    import __graft_entry__ as ge
    ge.build()
    from cfnerf_b200 import _lib
    lib = _lib.load()
    p = C.c_void_p(4096)
    args = [p, p, 4, 128, p, p, 256, p, 11, p, p, 0, p, p, p, None, None]
    assert lib.cfn_network_fwd_composite(None, *args) == CFN_EINVAL
    assert lib.cfn_network_fwd_composite(p, None, None, 4, 128, None, None, 0, None, 11, None, None, 0, None, None, None,
                                         None, None) == CFN_EINVAL


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
_NETS = {}


def _engine(cf, dev, K, variant, precision):
    key = (K, variant, precision)
    if key not in _NETS:
        cfg = O.CfnConfig(K=K)
        p = O.make_params(cfg, 0, variant)
        sa, sr = O.make_latents(cfg, 0)
        net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, sa, sr).to(dev)
        _NETS[key] = (net, cf.engine_for(net, dev, precision))
    return _NETS[key]


def _both(cf, dev, eng, net, B, N, white, kstats, seed):
    rays = O.synthetic_rays(B, seed).to(dev)
    g = torch.Generator().manual_seed(seed)
    t_rand = torch.rand(B, N, generator=g).to(dev)
    z = eng.zvals(rays, cf.reference_t_schedule(N, dev), t_rand, False)
    ea, er = cf.test_latents(net, dev)
    with torch.no_grad():
        fp = eng.network(B, N, rays=rays, z_vals=z)
        ref = eng.flow_composite(fp, z, rays[:, 3:6], 11, ea, er, white, want_kstats=kstats)
        out = eng.network(B, N, rays=rays, z_vals=z, composite=dict(rays_d=rays[:, 3:6], rays_d_stride=11, eps_alpha=ea,
                                                                    eps_rgb=er, white_bkgd=white, want_kstats=kstats))
    torch.cuda.synchronize()
    return ref, out


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp16", "bf16"])
@pytest.mark.parametrize("K", [1, 16, 32, 40, 128])
@pytest.mark.parametrize("N", [32, 64, 128])
def test_fused_is_bitwise_equal_to_network_then_flow_composite(precision, K, N):
    import cfnerf_b200 as cf
    dev = torch.device("cuda:0")
    # B * N never a multiple of 256; B = 1 and 37 leave most CTAs without a tile, 3001 walks many tiles per CTA
    cases = [(37, False, False), (37, True, False), (37, False, True), (37, True, True), (1, True, True), (3001, False, True)]
    for variant in ("default", "lively"):
        net, eng = _engine(cf, dev, K, variant, precision)
        for i, (B, white, kstats) in enumerate(cases):
            ref, out = _both(cf, dev, eng, net, B, N, white, kstats, seed=10 + i)
            keys = ("rgb_map", "disp_map", "depth_map") + (("kstats",) if kstats else ())
            for k in keys:
                assert out[k].shape == ref[k].shape, (k, out[k].shape, ref[k].shape)
                assert torch.equal(out[k], ref[k]), (variant, B, white, kstats, k, (out[k] - ref[k]).abs().max().item())
            if not kstats:
                assert out["kstats"] is None


@pytest.mark.gpu
def test_render_rays_takes_the_fused_path_by_the_rule(monkeypatch):
    import cfnerf_b200 as cf
    from cfnerf_b200 import api
    from cfnerf_b200.engine import Engine
    dev = torch.device("cuda:0")
    cfg = O.CfnConfig(K=32)
    sa, sr = O.make_latents(cfg, 0)
    net = cf.NeRFFlowsParams.from_oracle_params(cfg, O.make_params(cfg, 0, "lively"), sa, sr).to(dev)
    fine = cf.NeRFFlowsParams.from_oracle_params(cfg, O.make_params(cfg, 1, "lively"), sa, sr).to(dev)
    rays = O.synthetic_rays(300, 3).to(dev)
    calls = []
    orig = Engine.network

    def spy(self, B, N, *a, **k):
        calls.append((self.precision, N, k.get("composite") is not None))
        return orig(self, B, N, *a, **k)

    monkeypatch.setattr(Engine, "network", spy)

    def run(**kw):
        calls.clear()
        out = cf.render_rays(rays, net, None, 64, False, False, K_samples=32, want_kstats=True, **kw)
        torch.cuda.synchronize()
        return out, list(calls)

    fused, c = run(precision="fp16", white_bkgd=True)
    assert c == [("fp16", 64, True)]
    _, c = run(precision="bf16")
    assert c == [("bf16", 64, True)]
    _, c = run(precision="tf32")
    assert c == [("tf32", 64, False)]
    _, c = run(precision="fp16", want_weights=True)
    assert c == [("fp16", 64, False)]
    _, c = run(precision="fp16", N_importance=64, network_fine=fine)       # coarse needs weights; fine N = 128
    assert c == [("fp16", 64, False), ("fp16", 128, True)]
    _, c = run(precision="fp16", N_importance=128, network_fine=fine)      # fine N = 192
    assert c == [("fp16", 64, False), ("fp16", 192, False)]
    # the same render with the fused path switched off: bitwise the same maps
    monkeypatch.setattr(api, "fused_composite", lambda *a: False)
    two, c = run(precision="fp16", white_bkgd=True)
    assert c == [("fp16", 64, False)]
    for k in ("rgb_map", "disp_map", "depth_map", "kstats"):
        assert torch.equal(fused[k], two[k]), k
