// C-ABI entry points (include/cfnerf_b200.h): handle lifetime, parameter table, argument checking and
// dispatch to the kernels.  No torch types, no hidden device allocation outside create/pack.
#include <stdarg.h>

#include "handle.h"

namespace cfn {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
}  // namespace cfn

using namespace cfn;

extern "C" const char* cfn_last_error(void) { return g_err; }
extern "C" int cfn_version(void) { return 101; }

static void add_slot(CfnHandle* h, const std::string& name, int rows, int cols) {
  ParamSlot s;
  s.name = name;
  s.rows = rows;
  s.cols = cols;
  s.numel = (int64_t)rows * cols;
  s.offset = h->n_floats;
  h->n_floats += s.numel;
  h->slots.push_back(s);
}
static int add_linear(CfnHandle* h, const std::string& name, int out_f, int in_f) {
  int idx = (int)h->slots.size();
  add_slot(h, name + ".weight", out_f, in_f);
  add_slot(h, name + ".bias", out_f, 1);
  return idx;
}

extern "C" int cfn_create(const CfnConfig* cfg, CfnHandle** out) {
  CFN_CHECK_ARG(cfg && out, "cfn_create: null argument");
  CFN_CHECK_ARG(cfg->D >= 3 && cfg->D <= 16, "netdepth %d unsupported (3..16)", cfg->D);
  CFN_CHECK_ARG(cfg->W >= 16 && cfg->W % 2 == 0, "netwidth %d unsupported", cfg->W);
  CFN_CHECK_ARG(cfg->L_pos >= 0 && cfg->L_pos <= 16 && cfg->L_dir >= 0 && cfg->L_dir <= 16, "multires unsupported");
  CFN_CHECK_ARG(cfg->h_alpha >= 1 && cfg->h_rgb >= 1, "h sizes must be positive");
  CFN_CHECK_ARG(cfg->F >= 1 && cfg->F <= 8, "n_flows %d unsupported (1..8)", cfg->F);
  CFN_CHECK_ARG(cfg->K >= 1 && cfg->K <= 1024, "K_samples %d unsupported", cfg->K);
  CFN_CHECK_ARG(cfg->precision >= CFN_PREC_FP32 && cfg->precision <= CFN_PREC_TF32, "unknown precision mode");
  CfnHandle* h = new CfnHandle();
  h->cfg = *cfg;
  h->in_pos = 3 + 6 * cfg->L_pos;
  h->in_dir = 3 + 6 * cfg->L_dir;
  h->PP = 18 * cfg->F;
  // skips=[netdepth/2] with true division (main:327): only an even depth produces an integer layer index
  h->skip = (cfg->D % 2 == 0 && cfg->D / 2 <= cfg->D - 2) ? cfg->D / 2 : -1;
  h->n_floats = 0;
  h->packed = false;
  h->tc = nullptr;
  h->tc_dirty = 0;
  h->deterministic = 0;
  h->det_scratch = nullptr;
  h->det_floats = 0;
  h->gemm_tc = (cfg->precision != CFN_PREC_FP32) ? 1 : 0;
  h->gp = (h->in_pos + 7) & ~7;
  h->gd = (h->in_dir + 7) & ~7;
  // bf16 storage of the layer-by-layer chain (training in CFN_PREC_BF16): every row stride / column offset must be a
  // multiple of 8 elements (16 bytes); other widths keep the fp32-storage tf32 chain
  h->chain_bf16 = (h->gemm_tc && cfg->precision == CFN_PREC_BF16 && cfg->W % 16 == 0 && cfg->h_alpha % 8 == 0 &&
                   cfg->h_rgb % 8 == 0) ? 1 : 0;
  h->wg = h->amA_g = h->amC_g = nullptr;
  const int W = cfg->W, F = cfg->F;
  add_slot(h, "alpha_mean", 1, 1);
  add_slot(h, "alpha_std", 1, 1);
  add_slot(h, "rgb_mean", 3, 1);
  add_slot(h, "rgb_std", 3, 1);
  for (int i = 0; i < cfg->D; ++i) {
    int fin = (i == 0) ? h->in_pos : ((h->skip >= 0 && i == h->skip + 1) ? W + h->in_pos : W);
    add_linear(h, "pts_linears." + std::to_string(i), W, fin);
  }
  h->s_views = add_linear(h, "views_linears.0", W / 2, W + h->in_dir);
  h->s_feat = add_linear(h, "feature_linear", W, W);
  h->s_halpha = add_linear(h, "h_alpha_linear", cfg->h_alpha, W);
  h->s_hrgb = add_linear(h, "h_rgb_linear", cfg->h_rgb, W / 2);
  h->s_frgb = add_linear(h, "flows_rgb.amor_d", F * 9, cfg->h_rgb);
  add_linear(h, "flows_rgb.amor_diag1.0", F * 3, cfg->h_rgb);
  add_linear(h, "flows_rgb.amor_diag2.0", F * 3, cfg->h_rgb);
  add_linear(h, "flows_rgb.amor_b", F * 3, cfg->h_rgb);
  h->s_falpha = add_linear(h, "flows_alpha.amor_d", F, cfg->h_alpha);
  add_linear(h, "flows_alpha.amor_diag1.0", F, cfg->h_alpha);
  add_linear(h, "flows_alpha.amor_diag2.0", F, cfg->h_alpha);
  add_linear(h, "flows_alpha.amor_b", F, cfg->h_alpha);

  // gather tables: packed record row -> (source linear, row, tanh?)   (models.py:366-385; SURVEY §3.3(4))
  const int fa = h->s_falpha, fc = h->s_frgb;
  for (int f = 0; f < F; ++f) h->gatherA.push_back({fa + 2, fa + 3, f, 1});   // d1[f] = tanh(amor_diag1)[0,f]
  for (int f = 0; f < F; ++f) h->gatherA.push_back({fa + 4, fa + 5, f, 1});   // d2[f]
  for (int f = 0; f < F; ++f) h->gatherA.push_back({fa + 6, fa + 7, f, 0});   // b[f]
  for (int f = 0; f < F; ++f) {
    auto D = [&](int i, int j) { return GatherRow{fc + 0, fc + 1, (i * 3 + j) * F + f, 0}; };
    auto d1 = [&](int i) { return GatherRow{fc + 2, fc + 3, i * F + f, 1}; };
    auto d2 = [&](int i) { return GatherRow{fc + 4, fc + 5, i * F + f, 1}; };
    auto bb = [&](int i) { return GatherRow{fc + 6, fc + 7, i * F + f, 0}; };
    // R1: upper triangle of D, tanh'ed diag1 on the diagonal
    h->gatherC.push_back(d1(0)); h->gatherC.push_back(D(0, 1)); h->gatherC.push_back(D(0, 2));
    h->gatherC.push_back(d1(1)); h->gatherC.push_back(D(1, 2)); h->gatherC.push_back(d1(2));
    // R2: upper triangle of D^T, tanh'ed diag2 on the diagonal
    h->gatherC.push_back(d2(0)); h->gatherC.push_back(D(1, 0)); h->gatherC.push_back(D(2, 0));
    h->gatherC.push_back(d2(1)); h->gatherC.push_back(D(2, 1)); h->gatherC.push_back(d2(2));
    h->gatherC.push_back(bb(0)); h->gatherC.push_back(bb(1)); h->gatherC.push_back(bb(2));
  }

  auto fail = [&](const char* what) {
    set_error("cfn_create: %s", what);
    cfn_destroy(h);
    return CFN_ECUDA;
  };
  // operand views: padded row strides, gap after gamma(p) in the skip layer
  h->wg_floats = 0;
  for (size_t i = 0; i < h->slots.size(); ++i) {
    const ParamSlot& sl = h->slots[i];
    WView v{nullptr, 0, 0, 0};
    h->wg_offset.push_back(h->wg_floats);
    const bool is_weight = sl.name.size() > 7 && sl.name.compare(sl.name.size() - 7, 7, ".weight") == 0;
    if (is_weight) {
      const bool skip_in = h->skip >= 0 && (int)i == h->s_pts(h->skip + 1, 0);
      v.gap_at = skip_in ? h->in_pos : sl.cols;
      v.gap = skip_in ? h->gp - h->in_pos : 0;
      v.ld = (sl.cols + v.gap + 7) & ~7;
      h->wg_floats += (int64_t)sl.rows * v.ld / (h->chain_bf16 ? 2 : 1);
    }
    h->wv.push_back(v);
  }
  h->w32 = h->amA = h->amA_b = h->amC = h->amC_b = h->tanh_flags = nullptr;
  h->gatherA_dev = h->gatherC_dev = nullptr;
  if (cudaMalloc(&h->w32, h->n_floats * sizeof(float)) != cudaSuccess) return fail("cudaMalloc(w32)");
  h->globals = h->w32;
  if (cudaMalloc(&h->wg, (h->wg_floats + 4) * sizeof(float)) != cudaSuccess) return fail("cudaMalloc(wg)");
  if (cudaMemset(h->wg, 0, (h->wg_floats + 4) * sizeof(float)) != cudaSuccess) return fail("cudaMemset(wg)");
  for (size_t i = 0; i < h->slots.size(); ++i)
    if (h->wv[i].ld) h->wv[i].p = h->wg + h->wg_offset[i];
  if (cudaMalloc(&h->amA, (size_t)3 * F * cfg->h_alpha * sizeof(float)) != cudaSuccess) return fail("cudaMalloc");
  if (cudaMalloc(&h->amA_b, (size_t)3 * F * sizeof(float)) != cudaSuccess) return fail("cudaMalloc");
  if (cudaMalloc(&h->amC, (size_t)15 * F * cfg->h_rgb * sizeof(float)) != cudaSuccess) return fail("cudaMalloc");
  if (cudaMalloc(&h->amC_b, (size_t)15 * F * sizeof(float)) != cudaSuccess) return fail("cudaMalloc");
  if (h->gemm_tc) {
    if (cudaMalloc(&h->amA_g, (size_t)3 * F * cfg->h_alpha * sizeof(float)) != cudaSuccess) return fail("cudaMalloc");
    if (cudaMalloc(&h->amC_g, (size_t)15 * F * cfg->h_rgb * sizeof(float)) != cudaSuccess) return fail("cudaMalloc");
  } else {
    h->amA_g = h->amA;
    h->amC_g = h->amC;
  }
  if (cudaMalloc(&h->tanh_flags, (size_t)h->PP * sizeof(float)) != cudaSuccess) return fail("cudaMalloc");
  if (cudaMalloc(&h->gatherA_dev, h->gatherA.size() * sizeof(GatherRow)) != cudaSuccess) return fail("cudaMalloc");
  if (cudaMalloc(&h->gatherC_dev, h->gatherC.size() * sizeof(GatherRow)) != cudaSuccess) return fail("cudaMalloc");
  std::vector<float> flags;
  for (auto& g : h->gatherA) flags.push_back((float)g.tanh);
  for (auto& g : h->gatherC) flags.push_back((float)g.tanh);
  if (cudaMemcpy(h->tanh_flags, flags.data(), flags.size() * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess ||
      cudaMemcpy(h->gatherA_dev, h->gatherA.data(), h->gatherA.size() * sizeof(GatherRow), cudaMemcpyHostToDevice) !=
          cudaSuccess ||
      cudaMemcpy(h->gatherC_dev, h->gatherC.data(), h->gatherC.size() * sizeof(GatherRow), cudaMemcpyHostToDevice) !=
          cudaSuccess)
    return fail("cudaMemcpy(tables)");
  if (cfg->precision == CFN_PREC_BF16 || cfg->precision == CFN_PREC_FP16) {
    int rc = tc_create(h);
    if (rc != CFN_OK) {
      cfn_destroy(h);
      return rc;
    }
  }
  *out = h;
  return CFN_OK;
}

extern "C" int cfn_destroy(CfnHandle* h) {
  if (!h) return CFN_OK;
  if (h->tc) tc_destroy(h);
  cudaFree(h->det_scratch);
  cudaFree(h->w32);
  cudaFree(h->wg);
  if (h->amA_g != h->amA) cudaFree(h->amA_g);
  if (h->amC_g != h->amC) cudaFree(h->amC_g);
  cudaFree(h->amA);
  cudaFree(h->amA_b);
  cudaFree(h->amC);
  cudaFree(h->amC_b);
  cudaFree(h->tanh_flags);
  cudaFree(h->gatherA_dev);
  cudaFree(h->gatherC_dev);
  delete h;
  return CFN_OK;
}

extern "C" int cfn_param_count(const CfnHandle* h) { return h ? (int)h->slots.size() : 0; }
extern "C" const char* cfn_param_name(const CfnHandle* h, int i) {
  if (!h || i < 0 || i >= (int)h->slots.size()) return nullptr;
  return h->slots[i].name.c_str();
}
extern "C" int64_t cfn_param_numel(const CfnHandle* h, int i) {
  if (!h || i < 0 || i >= (int)h->slots.size()) return -1;
  return h->slots[i].numel;
}
extern "C" int cfn_flow_param_width(const CfnHandle* h) { return h ? h->PP : 0; }

extern "C" int cfn_pack_weights(CfnHandle* h, const float* const* params, int n_params, void* stream) {
  CFN_CHECK_ARG(h && params, "cfn_pack_weights: null argument");
  CFN_CHECK_ARG(n_params == (int)h->slots.size(), "cfn_pack_weights: expected %d tensors, got %d",
                (int)h->slots.size(), n_params);
  for (int i = 0; i < n_params; ++i) CFN_CHECK_ARG(params[i] != nullptr, "cfn_pack_weights: tensor %d is null", i);
  cudaStream_t s = (cudaStream_t)stream;
  int rc = pack_fp32(h, params, s);
  if (rc != CFN_OK) return rc;
  // the tensor-core weight stream of the fused render kernel (K1) is rebuilt lazily, by the first cfn_network_fwd that
  // needs it: a training loop that re-packs after every optimiser step never pays for it (0.12 ms of a 1.9 ms step)
  if (h->tc) h->tc_dirty = 1;
  h->packed = true;
  return CFN_OK;
}

static constexpr int64_t kChainPassPoints = 262144;   // points per internal pass of the non-saving chain (~2.6 GB fp32)

extern "C" int cfn_workspace_bytes(const CfnHandle* h, int64_t n_points, int save_for_backward, size_t* out) {
  CFN_CHECK_ARG(h && out && n_points >= 0, "cfn_workspace_bytes: bad argument");
  if (h->tc && !save_for_backward) {
    *out = tc_workspace_bytes(h, n_points);
    return CFN_OK;
  }
  // the layer-by-layer chain without saved activations walks the points in passes of at most kChainPassPoints, so its
  // workspace is bounded whatever the caller's ray chunk is (the reference bounds memory with netchunk, main:47-64)
  if (!save_for_backward && n_points > kChainPassPoints) n_points = kChainPassPoints;
  *out = chain_workspace_floats(h, n_points, save_for_backward) * sizeof(float) + 256;
  return CFN_OK;
}

extern "C" int cfn_zvals_f32(const float* rays, const float* t_vals, const float* t_rand, int lindisp, float* z_vals,
                             int64_t B, int N, void* stream) {
  CFN_CHECK_ARG(rays && t_vals && z_vals && B >= 0 && N >= 1, "cfn_zvals_f32: bad argument");
  return launch_zvals(rays, t_vals, t_rand, lindisp, z_vals, B, N, (cudaStream_t)stream);
}

extern "C" int cfn_rays_from_pose_f32(int H, int W, double focal, const float* c2w_host, double near, double far, int ndc,
                                      double ndc_near, float* rays, void* stream) {
  CFN_CHECK_ARG(c2w_host && rays, "cfn_rays_from_pose_f32: null argument");
  return launch_rays_from_pose(H, W, focal, c2w_host, near, far, ndc, ndc_near, rays, (cudaStream_t)stream);
}

extern "C" int cfn_network_fwd(CfnHandle* h, const float* rays, const float* z_vals, const float* pts,
                               const float* viewdirs, int64_t B, int N, float* flow_params, void* workspace,
                               size_t workspace_bytes, int save_for_backward, void* stream) {
  CFN_CHECK_ARG(h && flow_params && B >= 0 && N >= 1, "cfn_network_fwd: bad argument");
  CFN_CHECK_ARG((pts && viewdirs) || (rays && z_vals), "cfn_network_fwd: need (pts, viewdirs) or (rays, z_vals)");
  if (!h->packed) {
    set_error("cfn_network_fwd: call cfn_pack_weights first");
    return CFN_ESTATE;
  }
  if (B == 0) return CFN_OK;
  size_t need = 0;
  cfn_workspace_bytes(h, B * N, save_for_backward, &need);
  if (workspace_bytes < need || (!workspace && need)) {
    set_error("cfn_network_fwd: workspace %zu bytes < required %zu", workspace_bytes, need);
    return CFN_ENOMEM;
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (h->tc && !save_for_backward) {
    if (h->tc_dirty) {
      int rc = tc_pack(h, s);
      if (rc != CFN_OK) return rc;
      h->tc_dirty = 0;
    }
    return tc_network_fwd(h, rays, z_vals, pts, viewdirs, B, N, flow_params, workspace, workspace_bytes, s);
  }
  if (save_for_backward || B * N <= kChainPassPoints)
    return chain_network_fwd(h, rays, z_vals, pts, viewdirs, B, N, flow_params, (float*)workspace, save_for_backward, s);
  // bounded-memory passes over whole rays (results are independent of the split: every point is independent)
  CFN_CHECK_ARG(N <= kChainPassPoints, "cfn_network_fwd: N = %d samples per ray is too large", N);
  const int64_t rays_per_pass = kChainPassPoints / N;
  for (int64_t b0 = 0; b0 < B; b0 += rays_per_pass) {
    const int64_t nb = (B - b0 < rays_per_pass) ? (B - b0) : rays_per_pass;
    int rc = chain_network_fwd(h, rays ? rays + b0 * 11 : nullptr, z_vals ? z_vals + b0 * N : nullptr,
                               pts ? pts + b0 * N * 3 : nullptr, viewdirs ? viewdirs + b0 * 3 : nullptr, nb, N,
                               flow_params + b0 * N * h->PP, (float*)workspace, 0, s);
    if (rc != CFN_OK) return rc;
  }
  return CFN_OK;
}

extern "C" int cfn_network_bwd(CfnHandle* h, const float* g_flow_params, int64_t B, int N, void* workspace,
                               size_t workspace_bytes, float* const* grads, int n_params, void* stream) {
  CFN_CHECK_ARG(h && g_flow_params && grads && workspace, "cfn_network_bwd: null argument");
  CFN_CHECK_ARG(n_params == (int)h->slots.size(), "cfn_network_bwd: expected %d tensors", (int)h->slots.size());
  size_t need = 0;
  cfn_workspace_bytes(h, B * N, 1, &need);
  if (workspace_bytes < need) {
    set_error("cfn_network_bwd: workspace %zu bytes < required %zu", workspace_bytes, need);
    return CFN_ENOMEM;
  }
  return chain_network_bwd(h, g_flow_params, B, N, (float*)workspace, grads, (cudaStream_t)stream);
}

extern "C" int cfn_flow_composite_fwd(CfnHandle* h, const float* flow_params, const float* z_vals,
                                      const float* rays_d, int rays_d_stride, const float* eps_alpha,
                                      const float* eps_rgb, int64_t eps_group_rays, int64_t B, int N, int white_bkgd,
                                      float* rgb_map, float* disp_map, float* depth_map, float* raw, float* weights,
                                      float* logdet_sums, float* kstats, float* trans, float* seg_sums, int n_segments,
                                      void* stream) {
  CFN_CHECK_ARG(!seg_sums || (logdet_sums && n_segments >= 1 && n_segments <= 64 && N % n_segments == 0),
                "cfn_flow_composite_fwd: seg_sums needs the training flavour and N %% n_segments == 0");
  CFN_CHECK_ARG(eps_group_rays >= 0, "cfn_flow_composite_fwd: negative eps_group_rays");
  CFN_CHECK_ARG(!trans || logdet_sums, "cfn_flow_composite_fwd: trans is written by the training flavour only (pass logdet_sums)");
  CFN_CHECK_ARG(h && B >= 0 && (B == 0 || (flow_params && z_vals && rays_d && eps_alpha && eps_rgb && rgb_map && disp_map && depth_map)),
                "cfn_flow_composite_fwd: null argument");
  if (!h->packed) {
    set_error("cfn_flow_composite_fwd: call cfn_pack_weights first");
    return CFN_ESTATE;
  }
  // training (log-det sums requested) and the fp32 check mode keep the accurate functions
  // one-MUFU transcendentals behind every tensor-core mode (render and training); the log of the log-det stays accurate
  const int fast = (h->cfg.precision != CFN_PREC_FP32) ? 1 : 0;
  return launch_flow_composite_fwd(fast, h->cfg.F, h->cfg.K, h->globals, flow_params, z_vals, rays_d, rays_d_stride,
                                   eps_alpha, eps_rgb, eps_group_rays, B, N, white_bkgd, rgb_map, disp_map, depth_map, raw,
                                   weights, logdet_sums, kstats, trans, seg_sums, n_segments, (cudaStream_t)stream);
}

static int flow_composite_bwd_impl(CfnHandle* h, const float* flow_params, const float* z_vals, const float* rays_d,
                                  int rays_d_stride, const float* eps_alpha, const float* eps_rgb, int64_t eps_group_rays,
                                  int64_t B, int N, int white_bkgd, const float* g_rgb_map, const float* g_depth_map,
                                  float g_logdet_alpha, float g_logdet_rgb, const float* g_logdet_dev, float* trans,
                                  int trans_valid, const float* seg_sums, int n_segments, float* g_flow_params,
                                  float* g_globals_partial, void* stream) {
  CFN_CHECK_ARG(h && flow_params && z_vals && rays_d && eps_alpha && eps_rgb && g_rgb_map && g_flow_params &&
                    g_globals_partial && trans,
                "cfn_flow_composite_bwd: null argument");
  CFN_CHECK_ARG(eps_group_rays >= 0, "cfn_flow_composite_bwd: negative eps_group_rays");
  if (!h->packed) {
    set_error("cfn_flow_composite_bwd: call cfn_pack_weights first");
    return CFN_ESTATE;
  }
  return launch_flow_composite_bwd(h->cfg.precision != CFN_PREC_FP32 ? 1 : 0, h->cfg.F, h->cfg.K, h->globals, flow_params,
                                   z_vals, rays_d, rays_d_stride, eps_alpha, eps_rgb, eps_group_rays, B, N, white_bkgd,
                                   g_rgb_map, g_depth_map, g_logdet_alpha, g_logdet_rgb, g_logdet_dev, trans, trans_valid,
                                   seg_sums, n_segments, g_flow_params, g_globals_partial, (cudaStream_t)stream);
}

extern "C" int cfn_flow_composite_bwd(CfnHandle* h, const float* flow_params, const float* z_vals,
                                      const float* rays_d, int rays_d_stride, const float* eps_alpha,
                                      const float* eps_rgb, int64_t eps_group_rays, int64_t B, int N, int white_bkgd,
                                      const float* g_rgb_map, const float* g_depth_map, float g_logdet_alpha,
                                      float g_logdet_rgb, float* trans, int trans_valid, const float* seg_sums,
                                      int n_segments, float* g_flow_params, float* g_globals_partial, void* stream) {
  return flow_composite_bwd_impl(h, flow_params, z_vals, rays_d, rays_d_stride, eps_alpha, eps_rgb, eps_group_rays, B, N,
                                 white_bkgd, g_rgb_map, g_depth_map, g_logdet_alpha, g_logdet_rgb, nullptr, trans,
                                 trans_valid, seg_sums, n_segments, g_flow_params, g_globals_partial, stream);
}

extern "C" int cfn_flow_composite_bwd_dev(CfnHandle* h, const float* flow_params, const float* z_vals,
                                          const float* rays_d, int rays_d_stride, const float* eps_alpha,
                                          const float* eps_rgb, int64_t eps_group_rays, int64_t B, int N, int white_bkgd,
                                          const float* g_rgb_map, const float* g_depth_map, const float* g_logdet_dev,
                                          float* trans, int trans_valid, const float* seg_sums, int n_segments,
                                          float* g_flow_params, float* g_globals_partial, void* stream) {
  CFN_CHECK_ARG(g_logdet_dev != nullptr, "cfn_flow_composite_bwd_dev: g_logdet_dev is null");
  return flow_composite_bwd_impl(h, flow_params, z_vals, rays_d, rays_d_stride, eps_alpha, eps_rgb, eps_group_rays, B, N,
                                 white_bkgd, g_rgb_map, g_depth_map, 0.f, 0.f, g_logdet_dev, trans, trans_valid, seg_sums,
                                 n_segments, g_flow_params, g_globals_partial, stream);
}

extern "C" int cfn_raw2outputs_f32(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                                   int white_bkgd, float* rgb_map, float* disp_map, float* weights,
                                   float* depth_map, int64_t B, int N, int K, void* stream) {
  CFN_CHECK_ARG(B >= 0, "cfn_raw2outputs_f32: negative batch");
  CFN_CHECK_ARG(B == 0 || (raw && z_vals && rays_d && rgb_map && disp_map && depth_map),
                "cfn_raw2outputs_f32: null argument");
  return launch_raw2outputs(raw, z_vals, rays_d, rays_d_stride, white_bkgd, rgb_map, disp_map, weights, depth_map, B,
                            N, K, (cudaStream_t)stream);
}

extern "C" int cfn_sample_pdf_f32(const float* bins, const float* weights, const float* u, float* samples,
                                  int32_t* below, int64_t B, int M, int Nf, void* stream) {
  CFN_CHECK_ARG(B >= 0 && (B == 0 || Nf == 0 || (bins && weights && u && samples)), "cfn_sample_pdf_f32: null argument");
  return launch_sample_pdf(bins, weights, u, samples, below, B, M, Nf, (cudaStream_t)stream);
}

extern "C" int cfn_merge_sorted_f32(const float* a, const float* b, float* out, int64_t B, int Na, int Nb,
                                    void* stream) {
  CFN_CHECK_ARG(B >= 0 && Na >= 0 && Nb >= 0, "cfn_merge_sorted_f32: negative size");
  CFN_CHECK_ARG(B == 0 || ((a || Na == 0) && (b || Nb == 0) && (out || Na + Nb == 0)), "cfn_merge_sorted_f32: null argument");
  return launch_merge_sorted(a, b, out, B, Na, Nb, (cudaStream_t)stream);
}

extern "C" int cfn_mean_over_k_f32(const float* w, float* out, int64_t rows, int K, void* stream) {
  CFN_CHECK_ARG(w && out && rows >= 0 && K >= 1, "cfn_mean_over_k_f32: bad argument");
  return launch_mean_over_k(w, out, rows, K, (cudaStream_t)stream);
}

extern "C" int cfn_debug_profile(CfnHandle* h, uint64_t* out_host, int n) {
  CFN_CHECK_ARG(h && out_host && n > 0, "cfn_debug_profile: bad argument");
  return tc_debug_profile(h, (unsigned long long*)out_host, n);
}

extern "C" int cfn_gemm_f32(int engine, const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs,
                            int64_t b_cs, float* C, int64_t c_rs, const float* bias, const float* aux, int64_t aux_rs,
                            int64_t M, int N, int64_t K, int epilogue, int accumulate, int split_k, int round_out,
                            void* stream) {
  CFN_CHECK_ARG(M >= 0 && N >= 0 && K >= 0, "cfn_gemm_f32: bad shape");
  if (M == 0 || N == 0) return CFN_OK;
  CFN_CHECK_ARG(A && B && C, "cfn_gemm_f32: null argument");
  CFN_CHECK_ARG(engine == 0 || engine == 1, "cfn_gemm_f32: unknown engine %d", engine);
  GemmArgs g{};
  g.A = A; g.a_rs = a_rs; g.a_cs = a_cs;
  g.B = B; g.b_rs = b_rs; g.b_cs = b_cs;
  g.C = C; g.c_rs = c_rs; g.bias = bias; g.aux = aux; g.aux_rs = aux_rs;
  g.M = M; g.N = N; g.K = K; g.epilogue = epilogue; g.accumulate = accumulate; g.split_k = split_k;
  if (engine == 0) return launch_sgemm(g, (cudaStream_t)stream);
  return launch_tgemm(g, round_out, (cudaStream_t)stream);
}

extern "C" int cfn_gemm_bf16(const void* A, int64_t a_rs, int64_t a_cs, const void* B, int64_t b_rs, int64_t b_cs, void* C,
                             int64_t c_rs, int c_bf16, const float* bias, const float* aux, uint32_t* mask_out,
                             const uint32_t* aux_bits, int64_t bits_ld, int64_t M, int N, int64_t K, int epilogue,
                             int split_k, float* rowsum, void* stream) {
  CFN_CHECK_ARG(M >= 0 && N >= 0 && K >= 0, "cfn_gemm_bf16: bad shape");
  if (M == 0 || N == 0) return CFN_OK;
  CFN_CHECK_ARG(A && B && C, "cfn_gemm_bf16: null argument");
  GemmArgs g{};
  g.A = (const float*)A; g.a_rs = a_rs; g.a_cs = a_cs;
  g.B = (const float*)B; g.b_rs = b_rs; g.b_cs = b_cs;
  g.C = (float*)C; g.c_rs = c_rs; g.bias = bias; g.aux = aux; g.aux_rs = 0;
  g.M = M; g.N = N; g.K = K; g.epilogue = epilogue; g.split_k = split_k;
  g.mask_out = mask_out; g.aux_bits = aux_bits; g.bits_ld = bits_ld; g.rowsum = rowsum;
  g.ab_bf16 = 1; g.c_bf16 = c_bf16;
  CFN_CHECK_ARG(tgemm_supported(g), "cfn_gemm_bf16: operand layout / epilogue flavour not supported");
  CFN_CHECK_ARG(!rowsum || tgemm_can_rowsum(g), "cfn_gemm_bf16: rowsum needs split_k > 1 and at most one work item per CTA");
  return launch_tgemm(g, 0, (cudaStream_t)stream);
}

extern "C" int cfn_kde_nll_f32(const float* rgb_map, const float* target, int64_t B, int K, float grad_scale, float* partial,
                               float* g_rgb_map, void* stream) {
  CFN_CHECK_ARG(B >= 0 && (B == 0 || (rgb_map && target && partial)), "cfn_kde_nll_f32: null argument");
  return launch_kde_nll(rgb_map, target, B, K, grad_scale, partial, g_rgb_map, (cudaStream_t)stream);
}

extern "C" int cfn_trainer_loss_f32(const float* rgb_map, const float* depth_map, const float* target_rgb,
                                    const float* target_depth, int64_t B_rgb, int64_t B_depth, int K, float nll_scale,
                                    float depth_scale, float* partial, float* g_rgb_map, float* g_depth_map, void* stream) {
  CFN_CHECK_ARG(B_rgb >= 0 && B_depth >= 0, "cfn_trainer_loss_f32: negative batch");
  CFN_CHECK_ARG(B_rgb + B_depth == 0 || (rgb_map && depth_map && partial), "cfn_trainer_loss_f32: null argument");
  CFN_CHECK_ARG(B_rgb == 0 || target_rgb, "cfn_trainer_loss_f32: target_rgb is null");
  CFN_CHECK_ARG(B_depth == 0 || target_depth, "cfn_trainer_loss_f32: target_depth is null");
  return launch_trainer_loss(rgb_map, depth_map, target_rgb, target_depth, B_rgb, B_depth, K, nll_scale, depth_scale, partial,
                             g_rgb_map, g_depth_map, (cudaStream_t)stream);
}

extern "C" int cfn_adam_step_f32(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                                 float* const* exp_avg_sq, const int64_t* numels, float lr, float beta1, float beta2,
                                 float eps, int step, float grad_scale, void* stream) {
  CFN_CHECK_ARG(n_tensors == 0 || (params && grads && exp_avg && exp_avg_sq && numels), "cfn_adam_step_f32: null argument");
  return launch_adam(n_tensors, params, grads, exp_avg, exp_avg_sq, numels, lr, beta1, beta2, eps, step, grad_scale,
                     (cudaStream_t)stream);
}

extern "C" int cfn_adam_step_dev_f32(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                                     float* const* exp_avg_sq, const int64_t* numels, float* state_dev, float lr0,
                                     float decay_rate, float decay_steps, float beta1, float beta2, float eps,
                                     float grad_scale, void* stream) {
  CFN_CHECK_ARG(n_tensors == 0 || (params && grads && exp_avg && exp_avg_sq && numels), "cfn_adam_step_dev_f32: null argument");
  CFN_CHECK_ARG(state_dev != nullptr, "cfn_adam_step_dev_f32: state_dev is null");
  return launch_adam_dev(n_tensors, params, grads, exp_avg, exp_avg_sq, numels, state_dev, lr0, decay_rate, decay_steps, beta1,
                         beta2, eps, grad_scale, (cudaStream_t)stream);
}

extern "C" int cfn_globals_grad_f32(const CfnHandle* h, const float* g_globals_partial, int64_t B, float entropy_coef,
                                    float* out8, void* stream) {
  CFN_CHECK_ARG(h && g_globals_partial && out8 && B >= 0, "cfn_globals_grad_f32: bad argument");
  if (!h->packed) {
    set_error("cfn_globals_grad_f32: call cfn_pack_weights first");
    return CFN_ESTATE;
  }
  return launch_globals_grad(g_globals_partial, B, h->globals, entropy_coef, out8, (cudaStream_t)stream);
}

extern "C" int cfn_set_deterministic(CfnHandle* h, int on) {
  CFN_CHECK_ARG(h != nullptr, "cfn_set_deterministic: null handle");
  if (on && !h->det_scratch) {
    // the largest (splits x (out x in + out)) over every weight gradient the backward chain issues; the split count is
    // bounded by one K slice per CTA (tensor-core engine) or 8 per SM (CUDA-core engine), whichever engine runs
    int64_t need = 0;
    auto account = [&](int64_t out_f, int64_t in_f) {
      const int cg = out_f <= 128 ? 1 : 2;
      const int64_t bn = in_f >= 256 ? 256 : ((in_f + 15) / 16) * 16;
      const int64_t tiles_tc = ((out_f + 128 * cg - 1) / (128 * cg)) * ((in_f + bn - 1) / bn);
      const int64_t tiles_cc = ((out_f + 127) / 128) * ((in_f + 127) / 128);
      int64_t split = (148 / cg) / tiles_tc;
      const int64_t split_cc = (148 * 8 + tiles_cc - 1) / tiles_cc;
      if (split_cc > split) split = split_cc;
      if (split < 2) split = 2;
      const int64_t n = split * (out_f * in_f + out_f);
      if (n > need) need = n;
    };
    for (size_t i = 0; i < h->slots.size(); ++i)
      if (h->wv[i].ld) account(h->slots[i].rows, h->wv[i].ld);
    account(3 * h->cfg.F, (h->cfg.h_alpha + 7) & ~7);
    account(15 * h->cfg.F, (h->cfg.h_rgb + 7) & ~7);
    CFN_CUDA(cudaMalloc(&h->det_scratch, (size_t)need * sizeof(float)));
    h->det_floats = need;
  }
  h->deterministic = on ? 1 : 0;
  return CFN_OK;
}
