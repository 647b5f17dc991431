"""Multi-GPU plumbing (SURVEY §8(e)): one process per GPU under torchrun, rays sharded in contiguous blocks.

Rendering needs no collective (rays are independent, the latent draws are per-k, not per-ray): every rank renders
its block and the results are, bit for bit, the rows of the unsharded result.  Training averages gradients with ONE
all-reduce over a single flat fp32 bucket per step (the reference's nn.DataParallel instead re-broadcasts all
weights and scatters/gathers activations on every network call, run_nerf_uncertainty_NF.py:330).
"""
from __future__ import annotations

import torch
import torch.distributed as dist


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_bounds(n: int, rank: int, world_size: int):
    """Contiguous block [lo, hi) of rank `rank`; the first n % world ranks get one extra ray."""
    base, rem = divmod(n, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_rays(ray_batch: torch.Tensor, rank: int | None = None, world_size: int | None = None) -> torch.Tensor:
    r, w = world()
    rank = r if rank is None else rank
    world_size = w if world_size is None else world_size
    lo, hi = shard_bounds(ray_batch.shape[0], rank, world_size)
    return ray_batch[lo:hi]


def gather_rows(t: torch.Tensor, n_total: int) -> torch.Tensor:
    """All-gather the per-rank row blocks of a sharded render back into the full (n_total, ...) tensor."""
    rank, w = world()
    if w == 1:
        return t
    sizes = [hi - lo for lo, hi in (shard_bounds(n_total, r, w) for r in range(w))]
    biggest = max(sizes)                      # all_gather wants equal shapes: pad the short (ragged) blocks
    mine = t.contiguous()
    if mine.shape[0] < biggest:
        mine = torch.cat([mine, mine.new_zeros((biggest - mine.shape[0],) + tuple(t.shape[1:]))], 0)
    parts = [torch.empty_like(mine) for _ in range(w)]
    dist.all_gather(parts, mine)
    return torch.cat([p[:n] for p, n in zip(parts, sizes)], 0)


class GradBucket:
    """One flat fp32 bucket over every parameter that receives a gradient (the two dead heads alpha_linear /
    alpha_std_linear, models.py:59-60, have grad None and are left out: 2 359 520 of 2 360 546 elements)."""

    def __init__(self, params):
        self.params = [p for p in params if p.requires_grad]
        self.flat = None

    def _live(self):
        return [p for p in self.params if p.grad is not None]

    def all_reduce_mean_(self):
        rank, w = world()
        live = self._live()
        if w == 1 or not live:
            return
        n = sum(p.grad.numel() for p in live)
        if self.flat is None or self.flat.numel() != n or self.flat.device != live[0].grad.device:
            self.flat = torch.empty(n, dtype=torch.float32, device=live[0].grad.device)
        o = 0
        for p in live:
            k = p.grad.numel()
            self.flat[o:o + k].copy_(p.grad.reshape(-1))
            o += k
        dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)      # NCCL over NVLink on GPU tensors, gloo on CPU tensors
        self.flat.mul_(1.0 / w)
        o = 0
        for p in live:
            k = p.grad.numel()
            p.grad.copy_(self.flat[o:o + k].view_as(p.grad))
            o += k


def train_step(network_fn, optimizer, ray_batch, target, bucket: GradBucket | None = None, beta1: float = 0.01,
               depth_rays=None, target_depth=None, depth_lambda: float = 0.0, **render_kwargs):
    """One data-parallel optimisation step on this rank's shard (the trainer body of main:1014-1067 with the
    DataParallel wrapper replaced by one gradient all-reduce).  Equal shard sizes make the averaged gradient equal
    to the global-batch gradient of the mean-reduced loss.  `depth_rays` (Bd,11) / `target_depth` (Bd) add the
    depth-supervised rays of the shipped recipe (--colmap_depth, main:965-977, 1009-1011, 1018-1023, 1053-1054)."""
    from . import api

    rays = ray_batch if depth_rays is None else torch.cat([ray_batch, depth_rays], 0)             # main:1009-1011
    out = api.render_rays(rays, network_fn, None, 128, True, False, perturb=1., raw_noise_std=1., **render_kwargs)
    K = out["rgb_map"].shape[-1]
    losses = api.trainer_loss(out, target, K, beta1, target_depth=target_depth, depth_lambda=depth_lambda)
    optimizer.zero_grad(set_to_none=True)
    losses["loss"].backward()
    if bucket is not None:
        bucket.all_reduce_mean_()
    optimizer.step()
    return {k: v.detach() for k, v in losses.items()}


class FusedTrainStep:
    """The trainer body (main:1014-1067: render in train mode -> K-mean + KDE-NLL + beta1 * entropy [+ depth_lambda *
    depth MSE on the depth rays] -> backward -> Adam with the reference's lr decay) as a straight chain of C-ABI calls,
    without an autograd graph: cfn_zvals -> cfn_network_fwd(save) -> cfn_flow_composite_fwd (also writes the
    transmittances the backward reads) -> cfn_trainer_loss (loss + gradient seeds) -> cfn_flow_composite_bwd_dev ->
    cfn_network_bwd -> cfn_globals_grad -> [one all-reduce of the flat gradient] -> cfn_adam_step_dev -> cfn_pack_weights.

    Same kernels and numbers as `train_step`.  Parameters, gradients and Adam moments each live in ONE flat fp32 buffer
    (the module's Parameters are re-pointed at views of it: the gradient buffer is the all-reduce bucket, the weight
    re-pack is a single copy).  With `use_graph=True` the chain is captured once per batch shape into CUDA graphs and
    replayed: at the reference's own batch size (N_rand = 512 rays) a step is ~200 launches and ~80 tensor-map encodes
    of host work for ~1.5 ms of device work, so launch overhead is what bounds it.  The optimiser clock (step count,
    decayed learning rate) lives on the device so that it advances inside the graph."""

    def __init__(self, network_fn, lr: float = 5e-4, betas=(0.9, 0.999), eps: float = 1e-8, beta1: float = 0.01,
                 precision: str | None = None, N_samples: int = 128, white_bkgd: bool = False, lindisp: bool = False,
                 depth_lambda: float = 0.0, netchunk: int | None = None, lrate_decay: float = 0.0,
                 use_graph: bool = False, deterministic: bool = False):
        from . import api
        from .engine import _unwrap, engine_for
        self.module = _unwrap(network_fn)
        self.dev = next(self.module.parameters()).device
        self.eng = engine_for(network_fn, self.dev, precision or api.DEFAULT_TRAIN_PRECISION)
        self.lr, self.betas, self.eps, self.beta1 = lr, betas, eps, beta1
        self.N, self.white_bkgd, self.lindisp = N_samples, white_bkgd, lindisp
        self.depth_lambda = float(depth_lambda)
        self.netchunk = api.DEFAULT_NETCHUNK if netchunk is None else int(netchunk)
        self.decay_steps = float(lrate_decay) * 1000.0            # args.lrate_decay is in thousands of steps (main:1074)
        self.use_graph = bool(use_graph)
        if deterministic:       # two-pass split-K weight gradients: bitwise identical steps for identical inputs
            self.eng.set_deterministic(True)
        ps = self.eng.params
        n = sum(p.numel() for p in ps)
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.flat_param = torch.empty(n, **f32)
        self.flat_grad, self.exp_avg, self.exp_avg_sq = (torch.zeros(n, **f32) for _ in range(3))
        self.grads, self._m, self._v, o = [], [], [], 0
        with torch.no_grad():
            for p in ps:
                k = p.numel()
                view = self.flat_param[o:o + k].view(p.shape)
                view.copy_(p.detach())
                p.data = view                     # same Parameter object (optimizers / state_dict keep working)
                self.grads.append(self.flat_grad[o:o + k].view(p.shape))
                self._m.append(self.exp_avg[o:o + k])
                self._v.append(self.exp_avg_sq[o:o + k])
                o += k
        import ctypes as C
        arr = lambda ts: (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])  # noqa: E731
        self._arrs = (arr(ps), arr(self.grads), arr(self._m), arr(self._v), (C.c_int64 * len(ps))(*[p.numel() for p in ps]))
        self.adam_state = torch.zeros(4, **f32)    # [step, lr, 1 - b1^t, sqrt(1 - b2^t)] — advanced on the device
        self.step_count = 0
        self._shapes = {}

    # ---- static per-shape state -------------------------------------------------------------------------------
    def _buffers(self, B_rgb: int, B_depth: int):
        key = (B_rgb, B_depth)
        st = self._shapes.get(key)
        if st is not None:
            return st
        from . import api
        B, N, K, dev = B_rgb + B_depth, self.N, self.eng.K, self.dev
        f32 = dict(dtype=torch.float32, device=dev)
        group_rays, G = api.latent_groups(B, N, self.netchunk)
        st = dict(B=B, B_rgb=B_rgb, B_depth=B_depth, group_rays=group_rays, G=G,
                  rays=torch.empty(B, 11, **f32), target=torch.empty(B_rgb, 3, **f32),
                  target_depth=torch.empty(max(B_depth, 1), **f32), t_rand=torch.empty(B, N, **f32),
                  eps_a=torch.empty(G, K, **f32), eps_c=torch.empty(G, K, 3, **f32),
                  partial=torch.empty(B, 3, **f32), g_rgb=torch.empty(B, 3, K, **f32), g_depth=torch.empty(B, K, **f32),
                  graph_a=None, graph_b=None, out=None)
        # d loss / d (per-ray sum of log-dets) (models.py:286): the entropy term is the point-weighted mean of the per-call
        # scalars over ALL rows (main:1045) — or, with depth rays, over the first N_batch ROWS only (main:1023), which all
        # belong to the first network call: only its rays carry a seed, normalised by that call's own point count
        g_ld = torch.zeros(B, 2, **f32)
        if B_depth > 0:
            first = min(group_rays, B) if group_rays else B
            g_ld[:first] = -self.beta1 / float(first * N * K)
        else:
            g_ld[:] = -self.beta1 / float(B * N * K)
        st["g_ld"] = g_ld
        self._shapes[key] = st
        return st

    # ---- the chain --------------------------------------------------------------------------------------------
    def _forward_backward(self, st):
        from ._lib import check
        from .engine import _ptr, _stream
        eng, N, K = self.eng, self.N, self.eng.K
        B, rays = st["B"], st["rays"]
        from . import api
        t_vals = api.reference_t_schedule(N, self.dev)
        z = eng.zvals(rays, t_vals, st["t_rand"], self.lindisp)
        fp, ws = eng.network(B, N, rays=rays, z_vals=z, save=True)
        out = eng.flow_composite(fp, z, rays[:, 3:6], 11, st["eps_a"], st["eps_c"], self.white_bkgd, train=True,
                                 eps_group_rays=st["group_rays"], want_trans=True)
        Bd = st["B_depth"]
        check(eng.lib.cfn_trainer_loss_f32(_ptr(out["rgb_map"]), _ptr(out["depth_map"]), _ptr(st["target"]),
                                           _ptr(st["target_depth"]) if Bd else None, st["B_rgb"], Bd, K,
                                           1.0 / (3.0 * st["B_rgb"]), (self.depth_lambda / Bd) if Bd else 0.0,
                                           _ptr(st["partial"]), _ptr(st["g_rgb"]), _ptr(st["g_depth"]), _stream()),
              "cfn_trainer_loss_f32")
        g_fp, g_glob = eng.flow_composite_bwd(fp, z, rays[:, 3:6], 11, st["eps_a"], st["eps_c"], self.white_bkgd,
                                              st["g_rgb"], st["g_depth"] if Bd else None, st["g_ld"],
                                              trans=out["trans"], eps_group_rays=st["group_rays"],
                                              seg_sums=out["seg_sums"])
        eng.network_bwd(g_fp, B, N, ws, grads=self.grads)
        # parameters 0..3 (alpha_mean, alpha_std, rgb_mean, rgb_std) sit first in the flat gradient buffer
        check(eng.lib.cfn_globals_grad_f32(eng.h, _ptr(g_glob), g_glob.shape[0], float(self.beta1), _ptr(self.flat_grad),
                                           _stream()),
              "cfn_globals_grad_f32")
        st["out"] = out

    def _update(self, world: int):
        from ._lib import check
        from .engine import _ptr, _stream
        eng = self.eng
        p_arr, g_arr, m_arr, v_arr, numels = self._arrs
        check(eng.lib.cfn_adam_step_dev_f32(len(eng.params), p_arr, g_arr, m_arr, v_arr, numels, _ptr(self.adam_state),
                                            float(self.lr), 0.1, self.decay_steps, float(self.betas[0]),
                                            float(self.betas[1]), float(self.eps), 1.0 / world, _stream()),
              "cfn_adam_step_dev_f32")
        eng.pack(force=True)        # the next forward reads the re-packed operand copies

    @torch.no_grad()
    def step(self, ray_batch, target, t_rand=None, eps_alpha=None, eps_rgb=None, want_loss: bool = True,
             depth_rays=None, target_depth=None):
        from .engine import _f32c, bump_weights_epoch
        import math
        eng, dev, N, K = self.eng, self.dev, self.N, self.eng.K
        B_rgb = ray_batch.shape[0]
        B_depth = 0 if depth_rays is None else depth_rays.shape[0]
        rank, w = world()
        with torch.cuda.device(dev):
            st = self._buffers(B_rgb, B_depth)
            B, G = st["B"], st["G"]
            st["rays"][:B_rgb].copy_(ray_batch, non_blocking=True)
            st["target"].copy_(target, non_blocking=True)
            if B_depth:
                st["rays"][B_rgb:].copy_(depth_rays, non_blocking=True)                       # main:1009-1011
                st["target_depth"][:B_depth].copy_(target_depth, non_blocking=True)
            if t_rand is None:
                st["t_rand"].uniform_()                                                       # main:524
            else:
                st["t_rand"].copy_(t_rand, non_blocking=True)
            if eps_alpha is None:
                st["eps_a"].normal_()                                                         # models.py:234 (per call)
                st["eps_c"].normal_()                                                         # models.py:246
            else:
                st["eps_a"].copy_(_f32c(eps_alpha, dev).reshape(G, K))
                st["eps_c"].copy_(_f32c(eps_rgb, dev).reshape(G, K, 3))
            if not self.use_graph:
                self._forward_backward(st)
                if w > 1:
                    dist.all_reduce(self.flat_grad, op=dist.ReduceOp.SUM)
                self._update(w)
            elif st["graph_a"] is None:
                # first step of this shape: run it eagerly (warm-up: function attributes, allocator), then capture the same
                # calls for every later step.  The all-reduce stays outside the graphs (NCCL on the current stream).
                self._forward_backward(st)
                if w > 1:
                    dist.all_reduce(self.flat_grad, op=dist.ReduceOp.SUM)
                self._update(w)
                torch.cuda.synchronize()
                eager_out = st["out"]                # this step's results; the capture below re-binds st["out"]
                ga, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
                state_backup = [t.clone() for t in (self.flat_param, self.flat_grad, self.exp_avg, self.exp_avg_sq,
                                                    self.adam_state)]
                with torch.cuda.graph(ga):
                    self._forward_backward(st)
                with torch.cuda.graph(gb, pool=ga.pool()):
                    self._update(w)
                for t, bck in zip((self.flat_param, self.flat_grad, self.exp_avg, self.exp_avg_sq, self.adam_state),
                                  state_backup):
                    t.copy_(bck)          # capture does not execute, but keep the state provably untouched
                st["graph_a"], st["graph_b"] = ga, gb
                st["out_captured"], st["out"] = st["out"], eager_out
            else:
                if "out_captured" in st:
                    st["out"] = st.pop("out_captured")      # static tensors the replayed graph writes
                st["graph_a"].replay()
                if w > 1:
                    dist.all_reduce(self.flat_grad, op=dist.ReduceOp.SUM)
                st["graph_b"].replay()
            self.step_count += 1
            bump_weights_epoch()                          # other engines of this module re-pack on their next use ...
            eng._packed_version = eng._version()          # ... this one was re-packed inside the step
            if not want_loss:
                return {}
            from . import api
            out, partial = st["out"], st["partial"]
            tot = partial.sum(0)
            nll, mse = tot[0] / (3.0 * B_rgb), tot[1] / (3.0 * B_rgb)
            ent_rows = api._entropy_rows(self.module, st["eps_a"] if G > 1 else st["eps_a"][0],
                                         st["eps_c"] if G > 1 else st["eps_c"][0], out["logdet_sums"], B, N, K,
                                         st["group_rays"])
            ent = ent_rows[:B_rgb].mean() if B_depth else ent_rows.mean()                     # main:1023 / 1045
            res = {"loss_nll": nll, "mse": mse, "psnr": -10. * torch.log(mse) / math.log(10.), "loss_entropy": ent}
            loss = nll + self.beta1 * ent
            if B_depth:
                res["depth_loss"] = tot[2] / B_depth
                loss = loss + self.depth_lambda * res["depth_loss"]
            res["loss"] = loss
            return res

    def weights_checksum(self) -> torch.Tensor:
        """fp64 sum and sum of squares of the flat parameter buffer (ranks of a data-parallel job must agree bit for bit)."""
        p = self.flat_param.double()
        return torch.stack([p.sum(), (p * p).sum()])
