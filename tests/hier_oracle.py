"""Reference for ray gradients through the coarse+fine pass: `oracle.cfnerf_oracle.render_rays_hier` restated as one
autograd graph from the ray batch, following upstream nerf-pytorch's hierarchical step

    z_samples = sample_pdf(...).detach(); z_vals, _ = torch.sort(torch.cat([z_vals, z_samples], -1), -1)

The coarse depths keep their graph through a stable sort of cat[z_c, z_s]; the resampled depths z_s are constants.
`z_samples=` pins them (the library's own resampled depths, or a fixed set for finite differences); without it they
come from the oracle's sequential-fp32 sample_pdf exactly as render_rays_hier computes them, so the merged grid is
bitwise the oracle's numpy merge."""
import torch

from oracle import cfnerf_oracle as O


def merge_sorted_graph(z_c, z_s):
    """sort(cat[z_c, z_s]) with the graph of z_c kept and z_s a constant -> (z_all, src), src = the index into
    cat[z_c, z_s] of every slot (torch.sort(stable=True): ties keep the z_c-before-z_s order)."""
    cat = torch.cat([z_c, z_s.detach().to(z_c.dtype)], -1)
    _, src = torch.sort(cat.detach(), dim=-1, stable=True)
    return torch.gather(cat, -1, src), src


def render_rays_hier(p_coarse, p_fine, cfg, ray_batch, eps_alpha, eps_rgb, train, n_coarse, n_fine, t_rand=None, u=None,
                     lindisp=False, white_bkgd=False, faithful=False, z_samples=None):
    """O.render_rays_hier with ray gradients (the same outputs, plus "src")."""
    dtype = ray_batch.dtype
    rays_o, rays_d = ray_batch[:, 0:3], ray_batch[:, 3:6]
    viewdirs = ray_batch[:, -3:]
    near, far = ray_batch[:, 6:7], ray_batch[:, 7:8]
    B = ray_batch.shape[0]
    z_c = O.z_from_t(O.coarse_t_schedule(n_coarse, dtype), near, far, lindisp, t_rand)
    pts_c = rays_o[..., None, :] + rays_d[..., None, :] * z_c[..., :, None]
    raw_c, ents_c = O.run_network(p_coarse, cfg, pts_c, viewdirs, eps_alpha, eps_rgb, train, faithful=faithful)
    rgb0, disp0, w_c, depth0 = O.raw2outputs(raw_c, z_c, rays_d, white_bkgd)
    if z_samples is None:
        w_mean = w_c.mean(-1)
        z_mid = 0.5 * (z_c[..., 1:] + z_c[..., :-1])
        if u is None:
            u = torch.linspace(0.0, 1.0, steps=n_fine).expand(B, n_fine)
        z_s, _ = O.sample_pdf(z_mid.detach().float().numpy(), w_mean[..., 1:-1].detach().float().numpy(),
                              u.float().numpy())
        z_samples = torch.from_numpy(z_s)
    z_all, src = merge_sorted_graph(z_c, z_samples)
    pts_f = rays_o[..., None, :] + rays_d[..., None, :] * z_all[..., :, None]
    raw_f, ents_f = O.run_network(p_fine, cfg, pts_f, viewdirs, eps_alpha, eps_rgb, train, faithful=faithful)
    rgb_map, disp_map, w_f, depth_map = O.raw2outputs(raw_f, z_all, rays_d, white_bkgd)
    ret = {"rgb_map": rgb_map, "disp_map": disp_map, "depth_map": depth_map, "rgb0": rgb0, "disp0": disp0,
           "depth0": depth0, "z_vals": z_all, "z_samples": z_samples, "weights0": w_c, "src": src}
    if train:
        ret["loss_entropy"] = O.entropy_mean(ents_f)
        ret["loss_entropy0"] = O.entropy_mean(ents_c)
    return ret
