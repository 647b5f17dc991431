"""Engine: one C-ABI handle bound to one parameter-holding `network_fn` (the reference's `NeRF_Flows`, possibly
wrapped in `nn.DataParallel`, or `cfnerf_b200.network.NeRFFlowsParams`).  PyTorch here is plumbing only: device
memory, the stream and autograd bookkeeping; every number is produced by the CUDA library.
"""
from __future__ import annotations

import ctypes as C
import weakref

import torch

from . import _lib
from ._lib import CfnConfigC, check


def _unwrap(network_fn):
    return network_fn.module if hasattr(network_fn, "module") and isinstance(
        network_fn, torch.nn.DataParallel) else network_fn


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _f32c(t: torch.Tensor, device) -> torch.Tensor:
    if t.device != device or t.dtype != torch.float32:
        t = t.to(device=device, dtype=torch.float32)
    return t if t.is_contiguous() else t.contiguous()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def backward_segments(B: int, N: int) -> int:
    """Sample ranges per ray for the flow/compositing backward (one warp each).  A B200 holds 148 SMs x 16 warps of that
    kernel: below ~16k rays the ray count alone leaves slots empty or a ragged last wave (512 rays, the reference's batch:
    a fifth of the slots), so every ray is walked as 4 independent ranges."""
    return 4 if (B < 16384 and N % 16 == 0) else 1


_WEIGHTS_EPOCH = 0


def bump_weights_epoch():
    """Called by code that updates parameters without going through torch in-place ops (FusedAdam): every Engine
    re-packs its weights on its next use."""
    global _WEIGHTS_EPOCH
    _WEIGHTS_EPOCH += 1


class Engine:
    """Owns a CfnHandle for `module` on `device` at one precision mode ("fp32" | "bf16" | "fp16")."""

    def __init__(self, module, device, precision: str = "bf16"):
        if not torch.cuda.is_available():
            raise RuntimeError("cfnerf_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.module = weakref.ref(module)
        self.device = torch.device(device)
        self.precision = precision
        m = module
        L_pos, L_dir = (m.input_ch - 3) // 6, (m.input_ch_views - 3) // 6
        if 3 + 6 * L_pos != m.input_ch or 3 + 6 * L_dir != m.input_ch_views:
            raise ValueError("input_ch / input_ch_views must be 3+6L (get_embedder with include_input, helpers:54-69)")
        self.cfg = CfnConfigC(D=m.D, W=m.W, L_pos=L_pos, L_dir=L_dir, h_alpha=m.h_alpha_size, h_rgb=m.h_rgb_size,
                              F=m.n_flows, K=m.K_samples, precision=_lib.PREC[precision])
        self.K, self.F = m.K_samples, m.n_flows
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            check(self.lib.cfn_create(C.byref(self.cfg), C.byref(h)), "cfn_create")
        self.h = h
        self._finalizer = weakref.finalize(self, self.lib.cfn_destroy, h)
        self.PP = self.lib.cfn_flow_param_width(h)
        n = self.lib.cfn_param_count(h)
        self.names = [self.lib.cfn_param_name(h, i).decode() for i in range(n)]
        self.numels = [self.lib.cfn_param_numel(h, i) for i in range(n)]
        sd = dict(module.named_parameters())
        missing = [k for k in self.names if k not in sd]
        if missing:
            raise KeyError(f"network_fn lacks parameters {missing[:4]}...")
        self.params = [sd[k] for k in self.names]
        for p, ne, k in zip(self.params, self.numels, self.names):
            if p.numel() != ne:
                raise ValueError(f"{k}: {p.numel()} elements, expected {ne}")
            if p.device != self.device:
                raise ValueError(f"{k} lives on {p.device}, engine on {self.device}")
        self._packed_version = None
        self._ws = None

    def set_deterministic(self, on: bool = True):
        """Bitwise run-to-run stable weight gradients (two-pass split-K instead of fp32 atomics; cfn_set_deterministic)."""
        with torch.cuda.device(self.device):
            check(self.lib.cfn_set_deterministic(self.h, int(bool(on))), "cfn_set_deterministic")
        return self

    # ---- weights --------------------------------------------------------------------------------------
    def _version(self):
        return (_WEIGHTS_EPOCH,) + tuple(p._version for p in self.params) + tuple(p.data_ptr() for p in self.params)

    def pack(self, force: bool = False):
        """Re-pack the fp32 master weights when any parameter changed since the last call."""
        v = self._version()
        if not force and v == self._packed_version:
            return
        tensors = [_f32c(p.detach(), self.device) for p in self.params]
        arr = (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
        check(self.lib.cfn_pack_weights(self.h, arr, len(tensors), _stream()), "cfn_pack_weights")
        self._packed_version = v

    def workspace(self, n_points: int, save: bool):
        need = C.c_size_t()
        check(self.lib.cfn_workspace_bytes(self.h, n_points, int(save), C.byref(need)), "cfn_workspace_bytes")
        if save:  # saved activations belong to one autograd node: never share
            return torch.empty(need.value, dtype=torch.uint8, device=self.device)
        if self._ws is None or self._ws.numel() < need.value:
            self._ws = torch.empty(need.value, dtype=torch.uint8, device=self.device)
        return self._ws

    # ---- stages ---------------------------------------------------------------------------------------
    def zvals(self, rays, t_vals, t_rand, lindisp: bool):
        B, N = rays.shape[0], t_vals.numel()
        z = torch.empty(B, N, dtype=torch.float32, device=self.device)
        check(self.lib.cfn_zvals_f32(_ptr(rays), _ptr(t_vals), _ptr(t_rand), int(lindisp), _ptr(z), B, N, _stream()),
              "cfn_zvals_f32")
        return z

    def network(self, B: int, N: int, rays=None, z_vals=None, pts=None, viewdirs=None, save: bool = False,
                composite=None):
        """-> flow_params (B*N, 18F) [, workspace when save].
        composite=dict(rays_d=, rays_d_stride=, eps_alpha=, eps_rgb=, white_bkgd=, want_kstats=): the network and the
        render flavour of flow_composite in one kernel (cfn_network_fwd_composite; needs rays and z_vals) -> the dict
        flow_composite returns, bitwise equal to network() followed by flow_composite()."""
        self.pack()
        out = torch.empty(B * N, self.PP, dtype=torch.float32, device=self.device)
        ws = self.workspace(B * N, save)
        if composite is not None:
            K, f32 = self.K, dict(dtype=torch.float32, device=self.device)
            rgb, disp, depth = torch.empty(B, 3, K, **f32), torch.empty(B, K, **f32), torch.empty(B, K, **f32)
            ks = torch.empty(B, 8, **f32) if composite.get("want_kstats") else None
            c = composite
            check(self.lib.cfn_network_fwd_composite(self.h, _ptr(rays), _ptr(z_vals), B, N, _ptr(out), _ptr(ws), ws.numel(),
                                                     _ptr(c["rays_d"]), int(c["rays_d_stride"]), _ptr(c["eps_alpha"]),
                                                     _ptr(c["eps_rgb"]), int(bool(c["white_bkgd"])), _ptr(rgb), _ptr(disp),
                                                     _ptr(depth), _ptr(ks), _stream()), "cfn_network_fwd_composite")
            return dict(rgb_map=rgb, disp_map=disp, depth_map=depth, raw=None, weights=None, logdet_sums=None, kstats=ks,
                        trans=None, seg_sums=None)
        check(self.lib.cfn_network_fwd(self.h, _ptr(rays), _ptr(z_vals), _ptr(pts), _ptr(viewdirs), B, N, _ptr(out),
                                       _ptr(ws), ws.numel(), int(save), _stream()), "cfn_network_fwd")
        return (out, ws) if save else out

    def flow_composite(self, flow_params, z_vals, rays_d, rays_d_stride, eps_alpha, eps_rgb, white_bkgd: bool,
                       want_raw=False, want_weights=False, train=False, want_kstats=False, eps_group_rays: int = 0,
                       want_trans=False):
        """eps_alpha (K) / eps_rgb (K,3), or (G,K) / (G,K,3) with eps_group_rays = rays per latent-draw group.
        want_trans (training): also returns what the backward reads — `trans` (B,N,K) and, for batches small enough to
        leave warp slots empty, `seg_sums` (B,S,5,K) that let it walk S sample ranges of a ray in parallel."""
        self.pack()
        B, N = z_vals.shape
        K, dev = self.K, self.device
        f32 = dict(dtype=torch.float32, device=dev)
        rgb = torch.empty(B, 3, K, **f32)
        disp = torch.empty(B, K, **f32)
        depth = torch.empty(B, K, **f32)
        raw = torch.empty(B, N, K, 4, **f32) if want_raw else None
        w = torch.empty(B, N, K, **f32) if want_weights else None
        ld = torch.empty(B, 2, **f32) if train else None
        ks = torch.empty(B, 8, **f32) if want_kstats else None
        tr = torch.empty(B, N, K, **f32) if (train and want_trans) else None
        S = backward_segments(B, N) if tr is not None else 1
        sg = torch.empty(B, S, 5, K, **f32) if S > 1 else None
        check(self.lib.cfn_flow_composite_fwd(self.h, _ptr(flow_params), _ptr(z_vals), _ptr(rays_d), rays_d_stride,
                                              _ptr(eps_alpha), _ptr(eps_rgb), int(eps_group_rays), B, N, int(white_bkgd),
                                              _ptr(rgb), _ptr(disp), _ptr(depth), _ptr(raw), _ptr(w), _ptr(ld), _ptr(ks),
                                              _ptr(tr), _ptr(sg), S, _stream()), "cfn_flow_composite_fwd")
        return dict(rgb_map=rgb, disp_map=disp, depth_map=depth, raw=raw, weights=w, logdet_sums=ld, kstats=ks, trans=tr,
                    seg_sums=sg)

    def field_stats(self, flow_params, eps_alpha, eps_rgb, out=None):
        """flow_params (M,18F) from network(B=M, N=1, pts=, viewdirs=), base draws eps_alpha (K) / eps_rgb (K,3) ->
        (M,8) [sigma mean, sigma std, rgb mean (3), rgb std (3)] over the K draws (cfn_field_stats_f32; definitions in
        cfnerf_b200/field.py).  `out`: optional contiguous (M,8) fp32 device tensor to write into."""
        self.pack()
        M = flow_params.shape[0]
        if out is None:
            out = torch.empty(M, 8, dtype=torch.float32, device=self.device)
        check(self.lib.cfn_field_stats_f32(self.h, _ptr(flow_params), _ptr(eps_alpha), _ptr(eps_rgb), M, _ptr(out),
                                           _stream()), "cfn_field_stats_f32")
        return out

    def flow_composite_bwd(self,flow_params, z_vals, rays_d, rays_d_stride, eps_alpha, eps_rgb, white_bkgd,
                           g_rgb, g_depth, g_ld, *, trans, eps_group_rays: int = 0, seg_sums=None, ray_terms=False):
        """g_ld: device tensor (B,2) = d loss / d (per-ray sums of the alpha / rgb log-dets); stays on the device (no
        host sync).  trans / seg_sums: what the training forward (flow_composite(..., want_trans=True)) wrote.
        -> g_flow_params (B*N,18F), g_globals_partial (B*S,8) (sum the rows); with ray_terms also g_zdirect (B,N) and
        g_delta (B,N), the per-sample sums the ray gradient needs (cfn_flow_composite_bwd_rays)."""
        B, N = z_vals.shape
        S = seg_sums.shape[1] if seg_sums is not None else 1
        g_fp = torch.empty_like(flow_params)
        g_glob = torch.empty(B * S, 8, dtype=torch.float32, device=self.device)
        if ray_terms:
            g_zd = torch.empty(B, N, dtype=torch.float32, device=self.device)
            g_dl = torch.empty(B, N, dtype=torch.float32, device=self.device)
            check(self.lib.cfn_flow_composite_bwd_rays(
                self.h, _ptr(flow_params), _ptr(z_vals), _ptr(rays_d), rays_d_stride, _ptr(eps_alpha), _ptr(eps_rgb),
                int(eps_group_rays), B, N, int(white_bkgd), _ptr(g_rgb), _ptr(g_depth), _ptr(g_ld), _ptr(trans),
                _ptr(seg_sums), S, _ptr(g_fp), _ptr(g_glob), _ptr(g_zd), _ptr(g_dl), _stream()), "cfn_flow_composite_bwd_rays")
            return g_fp, g_glob, g_zd, g_dl
        check(self.lib.cfn_flow_composite_bwd(self.h, _ptr(flow_params), _ptr(z_vals), _ptr(rays_d), rays_d_stride,
                                              _ptr(eps_alpha), _ptr(eps_rgb), int(eps_group_rays), B, N, int(white_bkgd),
                                              _ptr(g_rgb), _ptr(g_depth), _ptr(g_ld), _ptr(trans), _ptr(seg_sums), S,
                                              _ptr(g_fp), _ptr(g_glob), _stream()),
              "cfn_flow_composite_bwd")
        return g_fp, g_glob

    def network_bwd(self, g_flow_params, B: int, N: int, ws, grads=None):
        """-> list of gradient tensors in parameter order (entries 0..3 are None: globals come from the flow stage).
        `grads`: optional preallocated fp32 tensors to write into (entries 0..3 ignored)."""
        if grads is None:
            grads = [None] * 4 + [torch.empty_like(p, dtype=torch.float32, memory_format=torch.contiguous_format)
                                  for p in self.params[4:]]
        arr = (C.c_void_p * len(grads))(*[(g.data_ptr() if (g is not None and i >= 4) else 0) for i, g in enumerate(grads)])
        check(self.lib.cfn_network_bwd(self.h, _ptr(g_flow_params), B, N, _ptr(ws), ws.numel(), arr, len(grads),
                                       _stream()), "cfn_network_bwd")
        return grads


    def network_bwd_inputs(self, g_flow_params, B: int, N: int, ws, weights: bool = True):
        """network_bwd that also returns g_enc (B*N, cfn_input_grad_width): the gradients of the encoded inputs
        (cfn_network_bwd_inputs).  weights=False: a frozen network, no weight gradient is computed -> (None, g_enc)."""
        g_enc = torch.empty(B * N, self.lib.cfn_input_grad_width(self.h), dtype=torch.float32, device=self.device)
        grads, arr = None, None
        if weights:
            grads = [None] * 4 + [torch.empty_like(p, dtype=torch.float32, memory_format=torch.contiguous_format)
                                  for p in self.params[4:]]
            arr = (C.c_void_p * len(grads))(*[(g.data_ptr() if (g is not None and i >= 4) else 0) for i, g in enumerate(grads)])
        check(self.lib.cfn_network_bwd_inputs(self.h, _ptr(g_flow_params), B, N, _ptr(ws), ws.numel(), arr, len(self.params),
                                              _ptr(g_enc), _stream()), "cfn_network_bwd_inputs")
        return grads, g_enc

    def ray_grad(self, rays, z_vals, t_vals, t_rand, lindisp: bool, g_enc, g_zdirect, g_delta, merged=None):
        """-> g_rays (B,11) = d loss / d [o d near far viewdir] (cfn_ray_grad_f32).  merged=(src, Nc): z_vals is the fine
        pass's merged grid, src (B,N) int32 its permutation (merge_sorted(..., return_src=True)) and t_vals / t_rand the
        coarse pass's (cfn_ray_grad_merged_f32)."""
        B, N = z_vals.shape
        out = torch.empty(B, 11, dtype=torch.float32, device=self.device)
        if merged is not None:
            src, Nc = merged
            check(self.lib.cfn_ray_grad_merged_f32(self.h, _ptr(rays), _ptr(z_vals), _ptr(src), int(Nc), _ptr(t_vals),
                                                   _ptr(t_rand), int(bool(lindisp)), _ptr(g_enc), _ptr(g_zdirect),
                                                   _ptr(g_delta), B, N, _ptr(out), _stream()), "cfn_ray_grad_merged_f32")
            return out
        check(self.lib.cfn_ray_grad_f32(self.h, _ptr(rays), _ptr(z_vals), _ptr(t_vals), _ptr(t_rand), int(bool(lindisp)),
                                        _ptr(g_enc), _ptr(g_zdirect), _ptr(g_delta), B, N, _ptr(out), _stream()),
              "cfn_ray_grad_f32")
        return out


_ENGINES: "weakref.WeakKeyDictionary" = weakref.WeakKeyDictionary()


def engine_for(network_fn, device=None, precision: str = "bf16") -> Engine:
    """Cached Engine per (module, device, precision)."""
    m = _unwrap(network_fn)
    if device is None:
        device = next(m.parameters()).device
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError(f"network_fn lives on {device}; cfnerf_b200 runs on CUDA only (no CPU fallback)")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    per = _ENGINES.setdefault(m, {})
    key = (str(device), precision)
    if key not in per:
        per[key] = Engine(m, device, precision)
    return per[key]
