"""CPU-side checks: the C-ABI library loads and exports every symbol include/cfnerf_b200.h declares; argument
validation fails cleanly without a GPU; the host mirror of the reference interface is consistent with the oracle."""
import ctypes as C
import os
import re

import pytest
import torch

from oracle import cfnerf_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from cfnerf_b200 import _lib
    return _lib.load()


def test_header_symbols_all_exported(lib):
    from cfnerf_b200 import _lib
    text = open(os.path.join(ROOT, "include", "cfnerf_b200.h")).read()
    declared = set(re.findall(r"\b(cfn_[a-z0-9_]+)\s*\(", text))
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in the header but not exported by the library"
    assert declared == set(_lib.SYMBOLS), "ctypes table and header disagree"


def test_invalid_config_is_rejected_without_touching_cuda(lib):
    from cfnerf_b200._lib import CfnConfigC
    cfg = CfnConfigC(D=1, W=512, L_pos=10, L_dir=4, h_alpha=64, h_rgb=64, F=4, K=32, precision=0)
    h = C.c_void_p()
    assert lib.cfn_create(C.byref(cfg), C.byref(h)) == -1
    assert b"netdepth" in lib.cfn_last_error()
    cfg = CfnConfigC(D=8, W=512, L_pos=10, L_dir=4, h_alpha=64, h_rgb=64, F=40, K=32, precision=0)
    assert lib.cfn_create(C.byref(cfg), C.byref(h)) == -1
    assert lib.cfn_version() >= 100


def test_no_cpu_fallback():
    """The product path refuses to run without its CUDA device instead of silently computing elsewhere."""
    import cfnerf_b200 as cf
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    net = cf.NeRFFlowsParams(netwidth=64, K_samples=4)
    with pytest.raises(RuntimeError):
        cf.render_rays(O.synthetic_rays(4), net, None, 128, False, False)
    with pytest.raises(RuntimeError):
        cf.raw2outputs(torch.zeros(1, 4, 2, 4), torch.zeros(1, 4), torch.zeros(1, 3))
    with pytest.raises(RuntimeError):
        net(torch.zeros(2, 90))
    with pytest.raises(RuntimeError):
        cf.render_rays_host(O.synthetic_rays(4), net, 128, K_samples=4)


def test_param_container_matches_reference_state_dict_layout():
    import cfnerf_b200 as cf
    for cfg in (O.CfnConfig(), O.CfnConfig(W=256, K=64, h_alpha=32)):
        p = O.make_params(cfg, 0)
        net = cf.NeRFFlowsParams.from_oracle_params(cfg, p, *O.make_latents(cfg, 0))
        sd = net.state_dict()
        assert set(sd) == set(p)
        for k in p:
            assert tuple(sd[k].shape) == tuple(p[k].shape), k
            assert torch.equal(sd[k], p[k])
        assert sum(v.numel() for v in sd.values()) == cfg.n_params()


def test_schedule_matches_oracle():
    import cfnerf_b200 as cf
    assert torch.equal(cf.reference_t_schedule(128, "cpu"), O.reference_t_schedule())
    assert torch.equal(cf.reference_t_schedule(64, "cpu"), O.coarse_t_schedule(64))


def test_kde_nll_loss_matches_oracle():
    import cfnerf_b200 as cf
    g = torch.Generator().manual_seed(0)
    rgb = torch.rand(16, 3, 32, generator=g)
    tgt = torch.rand(16, 3, generator=g)
    ent = torch.tensor(0.37)
    a = cf.kde_nll_loss(rgb, tgt, ent.expand(16 * 128, 32, 1), 32, 0.01)
    b = O.kde_nll_loss(rgb, tgt, ent, 32, 0.01)
    for k in a:
        assert abs(float(a[k]) - float(b[k])) <= 1e-6 * max(1.0, abs(float(b[k]))), k


def test_tf32_gemm_layout_contract_is_checked_on_the_host(lib):
    """cfn_gemm_f32 engine 1 (TMA-fed tcgen05 GEMM) refuses operand layouts the TMA cannot address — unit stride along
    one axis, 16-byte aligned bases and row strides — before any CUDA call is made (so this runs without a GPU)."""
    import ctypes as C

    def call(a_ptr, a_rs, a_cs, b_ptr, b_rs, b_cs, M=64, N=32, K=63, epi=0, split=1):
        return lib.cfn_gemm_f32(1, C.c_void_p(a_ptr), a_rs, a_cs, C.c_void_p(b_ptr), b_rs, b_cs, C.c_void_p(4096), N,
                                None, None, 0, M, N, K, epi, 0, split, 0, None)

    assert call(1024, 63, 1, 2048, 32, 1) == -1          # A row stride 63 floats: not a multiple of 16 bytes
    assert b"not supported" in lib.cfn_last_error()
    assert call(1028, 64, 1, 2048, 32, 1) == -1          # A base not 16-byte aligned
    assert call(1024, 64, 2, 2048, 32, 1) == -1          # no unit stride in A
    assert call(1024, 64, 1, 2048, 32, 1, epi=1) == -1   # ReLU epilogue is only instantiated for K-major B
    assert call(1024, 64, 1, 2048, 1, 64, split=4) == -1  # split-K (wgrad) needs M-major A and N-major B
    assert lib.cfn_gemm_f32(2, None, 0, 0, None, 0, 0, None, 0, None, None, 0, 4, 4, 4, 0, 0, 1, 0, None) == -1   # engine id


def test_latent_groups_follow_the_reference_batchify():
    """One latent draw per `batchify` call of netchunk points (main:47-64, models.py:233-251)."""
    from cfnerf_b200.api import latent_groups
    assert latent_groups(512, 128, 65536) == (0, 1)              # the shipped N_rand: exactly one call
    assert latent_groups(640, 128, 65536) == (512, 2)            # + 128 depth rays: a second call with its own noise
    assert latent_groups(4096, 128, 65536) == (512, 8)
    assert latent_groups(12, 128, 8 * 128) == (8, 2)
    assert latent_groups(4096, 192, 65536) == (0, 1)             # 192 does not divide netchunk: treated as one call
    # the oracle makes the same cut
    cfg = O.CfnConfig(W=64, D=4, K=4, h_alpha=16, h_rgb=16)
    p = O.make_params(cfg, 0, "lively")
    g = torch.Generator().manual_seed(0)
    ea, er = torch.randn(2, cfg.K, 1, generator=g), torch.randn(2, cfg.K, 3, generator=g)
    out = O.render_rays(p, cfg, O.synthetic_rays(12, 1), ea, er, True, t_rand=torch.rand(12, 128, generator=g),
                        faithful=False, netchunk=8 * 128)
    assert [n for _, n in out["entropy_calls"]] == [8 * 128, 4 * 128]


def test_backward_segments_and_defaults():
    from cfnerf_b200 import api
    from cfnerf_b200.engine import backward_segments
    assert backward_segments(512, 128) == 4 and backward_segments(4096, 128) == 4
    assert backward_segments(32768, 128) == 1 and backward_segments(512, 100) == 1
    old = (api.DEFAULT_PRECISION, api.DEFAULT_TRAIN_PRECISION, api.DEFAULT_NETCHUNK)
    try:
        api.configure(precision="tf32", netchunk=1024)
        assert api.DEFAULT_PRECISION == "tf32" and api.DEFAULT_NETCHUNK == 1024 and api.DEFAULT_TRAIN_PRECISION == old[1]
    finally:
        api.configure(*old)
    assert (api.DEFAULT_PRECISION, api.DEFAULT_TRAIN_PRECISION, api.DEFAULT_NETCHUNK) == old


def test_bench_workloads_and_flop_accounting():
    """bench.py's config table: the canonical network is 4 708 864 FLOP per point (SURVEY 8(d)); the three workloads have
    the shapes BASELINE.json names; the bench renders in a precision that passes every parity fixture."""
    import bench
    assert bench.flop_per_point(O.CfnConfig()) == 4708864
    assert bench.flop_per_point(O.CfnConfig(W=256, K=64, h_alpha=32)) == 1228544
    assert bench.RENDER_PRECISION in ("fp16", "tf32", "fp32")
    assert bench.image_rays_host("africa", 0).shape == (512 * 512, 11)
    r = bench.image_rays_host("fern", 0)
    assert r.shape == (1008 * 756, 11) and float(r[:, 6].max()) == 0.0 and float(r[:, 7].min()) == 1.0   # NDC near / far
    assert abs(float(r[0, 2]) + 1.0) < 1e-5                                                            # origins on the near plane
    p = bench.view_pose("lego", 50)
    assert abs(float(p[:, 3].norm()) - 4.0) < 1e-4                                                     # radius of pose_spherical


def test_bench_dump_outputs_sample_is_seeded_and_bounded(tmp_path):
    """bench.py --dump-outputs: the chunks of one step concatenated along the rays, float32; over the byte limit every
    array keeps the same seeded sample of rows, identical from run to run."""
    import numpy as np

    import bench
    g = torch.Generator().manual_seed(0)
    chunks = [{"rgb_map": torch.rand(n, 3, 4, generator=g), "depth_map": torch.rand(n, 4, generator=g),
               "kstats": torch.rand(n, 8, generator=g)} for n in (5, 7)]
    full = {k: torch.cat([c[k] for c in chunks], 0).numpy() for k in chunks[0]}
    assert bench.dump_outputs(str(tmp_path / "all"), chunks) == (12, 12)
    for k, v in full.items():
        a = np.load(tmp_path / "all" / f"{k}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, v), k
    per_ray = 4 * (12 + 4 + 8)
    limit = 4096 + 5 * per_ray
    dirs = [tmp_path / "a", tmp_path / "b"]
    for d in dirs:
        assert bench.dump_outputs(str(d), chunks, limit=limit) == (5, 12)
    assert sum(f.stat().st_size for f in dirs[0].iterdir()) <= limit
    rows = [int(np.nonzero((full["kstats"] == r).all(-1))[0][0]) for r in np.load(dirs[0] / "kstats.npy")]
    assert rows == sorted(set(rows)) and len(rows) == 5
    for k, v in full.items():
        a, b = np.load(dirs[0] / f"{k}.npy"), np.load(dirs[1] / f"{k}.npy")
        assert np.array_equal(a, b) and np.array_equal(a, v[rows]), k


def test_oracle_ref_staging_is_byte_identical():
    """oracle/_ref (git-ignored) is a byte-for-byte copy of the reference's *.py files when it exists."""
    from oracle import build_ref
    if not os.path.isfile(build_ref.MANIFEST):
        pytest.skip("oracle/_ref not staged")
    assert build_ref.check()
