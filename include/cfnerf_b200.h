/* cfnerf_b200 — C-ABI of the B200-native CF-NeRF render/train hot path.
 *
 * This header is the drop-in boundary (SURVEY.md §8(b)).  The reference (poetrywanderer/CF-NeRF) is pure
 * Python and has no FFI layer of its own; the callables a maintainer rebinds are
 *   run_nerf_uncertainty_NF.py:457-553  render_rays      -> cfn_zvals_f32 + cfn_network_fwd + cfn_flow_composite_fwd
 *   run_nerf_uncertainty_NF.py:67-85    run_network      -> cfn_network_fwd (+ cfn_flow_composite_fwd for raw)
 *   run_nerf_uncertainty_NF.py:411-454  raw2outputs      -> cfn_raw2outputs_f32
 *   run_nerf_helpers.py:9-11 (comment)  sample_pdf       -> cfn_sample_pdf_f32, cfn_merge_sorted_f32
 *   model/models.py:188-291             NeRF_Flows.forward / autograd backward -> *_fwd / *_bwd below
 * (cfnerf_b200/api.py holds the ctypes binding and the Python functions with the reference signatures;
 *  INTEGRATION.md shows the stub a maintainer adds to the reference.)
 *
 * Conventions: every function returns 0 on success and a negative CFN_E* code on failure, with a
 * thread-local message available from cfn_last_error().  All data pointers are DEVICE pointers owned by
 * the caller (fp32, row-major, contiguous unless a stride is passed); `stream` is a cudaStream_t passed as
 * void*; no function allocates device memory except cfn_create / cfn_pack_weights (handle-owned packed
 * weights).  Calls on one handle must be serialised by the caller; different handles are independent.
 * There is no CPU fallback anywhere behind this interface.
 */
#ifndef CFNERF_B200_H
#define CFNERF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CFN_OK 0
#define CFN_EINVAL (-1)   /* bad argument / unsupported configuration */
#define CFN_ECUDA (-2)    /* a CUDA runtime call or kernel launch failed */
#define CFN_ESTATE (-3)   /* call order violated (e.g. weights not packed) */
#define CFN_ENOMEM (-4)   /* workspace too small */

/* precision modes of the MLP chain (the only dense contraction on the path) */
#define CFN_PREC_FP32 0 /* CUDA-core fp32 FMA GEMMs: the 1e-5 "check" mode (render and training)                */
#define CFN_PREC_BF16 1 /* tcgen05.mma kind::f16, bf16 operands, fp32 accumulation in TMEM                  */
#define CFN_PREC_FP16 2 /* tcgen05.mma kind::f16, fp16 operands (11-bit significand, TF32-class), fp32 acc  */
#define CFN_PREC_TF32 3 /* tcgen05.mma kind::tf32 layer by layer, fp32 storage (operands rounded to tf32)       */
/* Training (cfn_network_fwd with save_for_backward + cfn_network_bwd) runs the layer-by-layer chain with saved
 * activations in every mode: fp32 FMA GEMMs in CFN_PREC_FP32; TMA-fed tcgen05 GEMMs otherwise — kind::f16 over
 * bf16-stored activations / gradients in CFN_PREC_BF16 (fp32 accumulation, master weights and weight gradients),
 * kind::tf32 over fp32 storage in CFN_PREC_TF32 and CFN_PREC_FP16. */

/* Architecture of one NeRF_Flows network (model/models.py:20-36; run_nerf_uncertainty_NF.py:317-336). */
typedef struct CfnConfig {
  int32_t D;        /* --netdepth          (8)   */
  int32_t W;        /* --netwidth          (512) */
  int32_t L_pos;    /* --multires          (10)  -> 3+6L = 63 input channels */
  int32_t L_dir;    /* --multires_views    (4)   -> 27 view channels         */
  int32_t h_alpha;  /* --h_alpha_size      (64)  */
  int32_t h_rgb;    /* --h_rgb_size        (64)  */
  int32_t F;        /* --n_flows           (4)   */
  int32_t K;        /* --K_samples         (32)  */
  int32_t precision; /* CFN_PREC_* */
} CfnConfig;

typedef struct CfnHandle CfnHandle;

const char* cfn_last_error(void);
int cfn_version(void);

/* ---- lifetime ------------------------------------------------------------------------------------ */
int cfn_create(const CfnConfig* cfg, CfnHandle** out);
int cfn_destroy(CfnHandle* h);

/* Opt-in bitwise run-to-run stable training gradients (SURVEY 7.3-5).  By default the split-K weight-gradient GEMMs of
 * cfn_network_bwd add their partial products with fp32 atomics, whose order varies between runs (differences ~1e-7
 * relative).  With on != 0 every K split stores its partial product into handle-owned scratch (allocated by this call,
 * like cfn_create / cfn_pack_weights: up to ~0.3 GB for the canonical network) and a second pass adds the slabs in split
 * order; the bias-gradient column sums use a fixed-order reduction as well.  Costs a few percent of a training step. */
int cfn_set_deterministic(CfnHandle* h, int on);

/* The parameter tensors the path reads, in the order cfn_pack_weights / cfn_network_bwd expect them.
 * Names are the keys of NeRF_Flows.state_dict() (model/models.py:38-67, 339-350); the two dead heads
 * alpha_linear / alpha_std_linear (models.py:59-60) are not part of the list. */
int cfn_param_count(const CfnHandle* h);
const char* cfn_param_name(const CfnHandle* h, int i);
int64_t cfn_param_numel(const CfnHandle* h, int i);

/* Copy/convert the fp32 master parameters into the handle's packed device layouts (fp32 gathered flow
 * conditioning matrices and GEMM operand copies; the bf16/fp16 pre-swizzled UMMA weight stream of the fused render
 * kernel is rebuilt from them by the next cfn_network_fwd that needs it, on that call's stream).
 * Call after every optimizer step.  params[i] is a device pointer to tensor i (fp32, contiguous). */
int cfn_pack_weights(CfnHandle* h, const float* const* params, int n_params, void* stream);

/* floats per 3-D point produced by the network stage: 18*F (alpha: d1,d2,b per flow; rgb: R1 (6), R2 (6), b (3) per flow) */
int cfn_flow_param_width(const CfnHandle* h);

/* ---- A1: sample schedule along each ray (run_nerf_uncertainty_NF.py:510-532) ------------------- */
/* rays (B,11) [o d near far viewdir]; t_vals (N) the [0,1] schedule; t_rand (B,N) stratified uniforms or
 * NULL (perturb == 0); writes z_vals (B,N) with the reference's fp32 operation order. */
int cfn_zvals_f32(const float* rays, const float* t_vals, const float* t_rand, int lindisp, float* z_vals,
                  int64_t B, int N, void* stream);

/* ---- F2: ray generation for a full image (render(..., c2w=pose), run_nerf_uncertainty_NF.py:129-158) ---------- */
/* c2w_host: 12 floats in HOST memory, the rows of c2w[:3,:4].  Writes rays (H*W,11) = [o d near far viewdir] on the
 * device: get_rays (run_nerf_helpers.py:288-297), viewdirs = d/|d| taken before the optional NDC warp
 * (ndc_rays(H,W,focal,ndc_near,...), helpers:360-377; the reference passes ndc_near = 1). */
int cfn_rays_from_pose_f32(int H, int W, double focal, const float* c2w_host, double near, double far, int ndc,
                           double ndc_near, float* rays, void* stream);

/* ---- A2-A5: positional encoding + MLP trunk/heads + flow conditioning ------------------------ */
/* Bytes of caller-provided workspace cfn_network_fwd needs for n_points points.
 * save_for_backward != 0 sizes it for the training path (activations kept for cfn_network_bwd).  Without saved
 * activations the layer-by-layer chain walks the points in internal passes of at most 262144 points, so the answer
 * is bounded whatever n_points is (the reference bounds its memory with netchunk, main:47-64). */
int cfn_workspace_bytes(const CfnHandle* h, int64_t n_points, int save_for_backward, size_t* out);

/* Points are either given explicitly (pts (B*N,3), run_network semantics, run_nerf_uncertainty_NF.py:67-85)
 * or, when pts == NULL, generated as o + d*z from rays (B,11) and z_vals (B,N) (main:534).
 * viewdirs (B,3) may be NULL when rays is given (columns 8..10 are used).
 * flow_params (B*N, 18F) receives the per-point conditional flow parameters (diagonals already tanh'ed). */
int cfn_network_fwd(CfnHandle* h, const float* rays, const float* z_vals, const float* pts, const float* viewdirs,
                    int64_t B, int N, float* flow_params, void* workspace, size_t workspace_bytes,
                    int save_for_backward, void* stream);

/* Render fast path (CFN_PREC_BF16 / CFN_PREC_FP16, n_flows = 4, N dividing 128, one latent-draw set for every ray):
 * cfn_network_fwd from (rays, z_vals) followed by the render flavour of cfn_flow_composite_fwd (no raw / weights /
 * log-dets), in ONE kernel whose spare warps composite each tile's rays while the network runs on the next tile.
 * flow_params (B*N,18F) is still written (and read back by the compositing warps).  Outputs are bitwise equal to
 * the two calls: rgb_map (B,3,K), disp_map (B,K), depth_map (B,K), kstats (B,8) optional. */
int cfn_network_fwd_composite(CfnHandle* h, const float* rays, const float* z_vals, int64_t B, int N, float* flow_params,
                              void* workspace, size_t workspace_bytes, const float* rays_d, int rays_d_stride,
                              const float* eps_alpha, const float* eps_rgb, int white_bkgd, float* rgb_map,
                              float* disp_map, float* depth_map, float* kstats, void* stream);

/* Backward of cfn_network_fwd (training path).  g_flow_params (B*N,18F) is d loss / d flow_params;
 * workspace must be the one a save_for_backward forward of the same points filled.  grads[i] (device,
 * fp32, same shapes/order as the parameters; entries may be NULL to skip) are OVERWRITTEN for i >= 4
 * (the four global latent parameters 0..3 get their gradient from cfn_flow_composite_bwd). */
int cfn_network_bwd(CfnHandle* h, const float* g_flow_params, int64_t B, int N, void* workspace,
                    size_t workspace_bytes, float* const* grads, int n_params, void* stream);

/* ---- A6-A8 (+A11 partials): K-sample flows + alpha compositing --------------------------------- */
/* eps_alpha (G,K), eps_rgb (G,K,3): base latent draws (models.py:198-206 / 233-251).  eps_group_rays = 0: G = 1, one
 * set shared by all rays (test mode; a training call of at most netchunk points).  eps_group_rays = R > 0: ray b uses
 * set b / R — the reference draws fresh noise in EVERY network call of netchunk points (batchify, main:47-64), i.e.
 * every netchunk / N rays of a training batch (512 rays at the shipped netchunk = 65536, N = 128).
 * rays_d: pointer to the first direction, rays_d_stride floats between rays (11 when it points into a ray batch).
 * Outputs: rgb_map (B,3,K), disp_map (B,K), depth_map (B,K); optional raw (B,N,K,4) [rgb|sigma],
 * weights (B,N,K); optional logdet_sums (B,2): per-ray sums over (n,k) of the alpha / rgb log-det terms
 * (models.py:263,278) for the entropy loss (requesting them selects the training flavour); optional kstats (B,8):
 * mean_k rgb (3), "uncertainty" std (unbiased std * K/(K-1), main:1034/1130) (3), mean_k depth, mean_k disp; optional
 * trans (B,N,K) (training flavour only): the transmittance in front of every sample, which cfn_flow_composite_bwd
 * reads; optional seg_sums (B, n_segments, 5, K) (training flavour only; N must be a multiple
 * of n_segments): per equal sample range of every ray the sums of w*rgb (3), w*z and w — they let the backward walk the
 * n_segments ranges of a ray in independent warps.  Any optional pointer may be NULL. */
int cfn_flow_composite_fwd(CfnHandle* h, const float* flow_params, const float* z_vals, const float* rays_d,
                           int rays_d_stride, const float* eps_alpha, const float* eps_rgb, int64_t eps_group_rays,
                           int64_t B, int N, int white_bkgd, float* rgb_map, float* disp_map, float* depth_map,
                           float* raw, float* weights, float* logdet_sums, float* kstats, float* trans, float* seg_sums,
                           int n_segments, void* stream);

/* Backward (SURVEY.md Appendix A).  g_rgb_map (B,3,K) and g_depth_map (B,K) (NULL = zero) are upstream
 * gradients.  g_logdet (B,2), REQUIRED, holds PER-RAY gradient seeds d loss / d(sum of log-dets) in DEVICE memory:
 * [b][0] = alpha, [b][1] = rgb (e.g. -beta1/(B*N*K)).  The host does not have to wait for the loss graph before it
 * issues the backward (no device-to-host sync per step), and rays of different network calls / loss terms can carry
 * different seeds (the depth rays of the shipped recipe take no part in the entropy term, main:1018-1023, 1045).
 * trans (B,N,K), REQUIRED: what cfn_flow_composite_fwd wrote for the same inputs.
 * seg_sums / n_segments: what cfn_flow_composite_fwd wrote for the same inputs (NULL / 1: one warp walks the whole ray;
 * n_segments > 1 gives small batches n_segments times the parallelism — the reference trains on 512 rays per step).
 * Writes g_flow_params (B*N,18F) and g_globals_partial (B*n_segments,8): per ray and range the
 * partial sums of d/d[alpha_mean, alpha_std, rgb_mean(3), rgb_std(3)] through z0 = eps*std+mean only (the caller sums
 * the rows; kept apart so the result is deterministic). */
int cfn_flow_composite_bwd(CfnHandle* h, const float* flow_params, const float* z_vals, const float* rays_d,
                           int rays_d_stride, const float* eps_alpha, const float* eps_rgb, int64_t eps_group_rays,
                           int64_t B, int N, int white_bkgd, const float* g_rgb_map, const float* g_depth_map,
                           const float* g_logdet, const float* trans, const float* seg_sums, int n_segments,
                           float* g_flow_params, float* g_globals_partial, void* stream);

/* ---- A8 stand-alone: raw2outputs (run_nerf_uncertainty_NF.py:411-454) ------------------------ */
int cfn_raw2outputs_f32(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride,
                        int white_bkgd, float* rgb_map, float* disp_map, float* weights, float* depth_map,
                        int64_t B, int N, int K, void* stream);

/* ---- A9: hierarchical resampling (extension; oracle/cfnerf_oracle.py sample_pdf) ------------ */
/* bins (B,M), weights (B,M-1), u (B,Nf) -> samples (B,Nf), optional below (B,Nf) int32.  Bit-exact with
 * the sequential-fp32 oracle. */
int cfn_sample_pdf_f32(const float* bins, const float* weights, const float* u, float* samples, int32_t* below,
                       int64_t B, int M, int Nf, void* stream);
/* out (B,Na+Nb) = sort(cat[a (B,Na), b (B,Nb)]) per row (values only). */
int cfn_merge_sorted_f32(const float* a, const float* b, float* out, int64_t B, int Na, int Nb, void* stream);
/* cfn_merge_sorted_f32 that also writes src (B,Na+Nb) int32: the index into cat[a, b] of every output slot (ties keep
 * the a-before-b order, i.e. torch.sort(stable=True)); out holds the same values bit for bit.  The permutation a ray
 * gradient on a merged grid needs (cfn_ray_grad_merged_f32, F7).  Detected by the symbol (cfn_version() stays 103). */
int cfn_merge_sorted_src_f32(const float* a, const float* b, float* out, int32_t* src, int64_t B, int Na, int Nb,
                             void* stream);
/* mean over K of weights (B,N,K) -> (B,N)  (the shared fine grid decision, SURVEY.md A9) */
int cfn_mean_over_k_f32(const float* w, float* out, int64_t rows, int K, void* stream);

/* ---- F1: K-reduction + KDE negative log-likelihood of the trainer (run_nerf_uncertainty_NF.py:1018-1055) ------ */
/* The whole loss of the shipped recipe (--colmap_depth, --depth_lambda) over the concatenated batch [B_rgb colour rays |
 * B_depth depth rays] (main:1009-1011) in one launch.  rgb_map (B,3,K), depth_map (B,K) with B = B_rgb + B_depth;
 * target_rgb (B_rgb,3); target_depth (B_depth) (depth_map and target_depth may be NULL when B_depth = 0).
 * partial (B,3) = per-ray [sum_c nll_c, sum_c (mean_k rgb - target)^2, (mean_k depth - target_depth)^2] (colour rays fill
 * columns 0-1, depth rays column 2).  g_rgb_map (B,3,K) = nll_scale * d(sum_c nll_c)/d rgb_map on colour rays (bandwidth
 * detached as in main:1036), 0 on depth rays (rgbs[:N_batch], main:1021); g_depth_map (B,K) = depth_scale *
 * d(err^2)/d depth_map on depth rays, 0 on colour rays; either may be NULL when not wanted.  The trainer's loss_nll is
 * sum(partial[:,0]) / (3 B_rgb): pass nll_scale = 1/(3 B_rgb) and depth_scale = depth_lambda / B_depth to seed the
 * backward directly. */
int cfn_trainer_loss_f32(const float* rgb_map, const float* depth_map, const float* target_rgb, const float* target_depth,
                         int64_t B_rgb, int64_t B_depth, int K, float nll_scale, float depth_scale, float* partial,
                         float* g_rgb_map, float* g_depth_map, void* stream);

/* ---- F5: evaluation of the predictive uncertainty (PSNR, KDE-NLL, AUSE; INTEGRATION.md §2) ----------------------- */
/* Per-pixel records of B rays from what K2 (kstats (B,8)) and cfn_trainer_loss_f32 (partial (B,3), B_rgb = B) wrote for
 * the same maps, target_rgb (B,3):  uncertainty = (s_0^2 + s_1^2 + s_2^2) / 3 with s the "uncertainty" std of kstats;
 * sq_err = partial[:,1] / 3; abs_err = mean_c |mean_k rgb - target|; nll = partial[:,0] / 3 (the KDE-NLL averaged over
 * the channels).  depth_map (B,K) may be NULL; when given, target_depth (B) is required and depth_uncertainty = unbiased
 * variance over k, depth_sq_err / depth_abs_err = squared / absolute error of mean_k depth.  K >= 2. */
int cfn_eval_records_f32(const float* kstats, const float* partial, const float* target_rgb, const float* depth_map,
                         const float* target_depth, int64_t B, int K, float* uncertainty, float* sq_err, float* abs_err,
                         float* nll, float* depth_uncertainty, float* depth_sq_err, float* depth_abs_err, void* stream);

/* Sparsification curves and AUSE of n_views views of n_pixels pixels each (1 <= n_views <= 65535, n_views * n_pixels
 * < 2^31, n_fractions = S >= 2).  uncertainty, sq_err and abs_err are (V,P) and must be finite and >= 0 (device
 * pointers: not checked).  For i < S, m_i = P - floor(i P / S) pixels are kept, the least uncertain first (stable: ties
 * keep the lower pixel index).  curves (V,4,S): [RMSE by uncertainty, RMSE oracle (by sq_err), MAE by uncertainty, MAE
 * oracle (by abs_err)], each divided by its value at i = 0 (0 when that is 0); ause (V,2) [RMSE, MAE] =
 * sum_{i<S-1} (d_i + d_{i+1}) / (2S), d = curve - oracle.  Bitwise deterministic.  workspace: at least
 * cfn_sparsification_workspace_bytes (which asks CUB for its temporary storage) bytes of device memory, else CFN_ENOMEM. */
int cfn_sparsification_workspace_bytes(int64_t n_views, int64_t n_pixels, int n_fractions, size_t* out);
int cfn_sparsification_f32(const float* uncertainty, const float* sq_err, const float* abs_err, int64_t n_views,
                           int64_t n_pixels, int n_fractions, void* workspace, size_t workspace_bytes, float* curves,
                           float* ause, void* stream);

/* ---- F6: field-space statistics over the K latent draws (INTEGRATION.md §2) ------------------------------------- */
/* For M query points whose flow records flow_params (M, 18F) cfn_network_fwd wrote (explicit points: B = M, N = 1),
 * run both flow stacks for the K base draws eps_alpha (K) / eps_rgb (K,3) and reduce over k on the device:
 * out (M,8) = [mean sigma, std sigma, mean rgb (3), std rgb (3)] with sigma_k = softplus(raw alpha) (main:424),
 * rgb_k = sigmoid(raw rgb) (main:431), std = sqrt(sum_k (x_k - mean)^2 / (K-1)) and 0 when K = 1 (the plain sample
 * std, not the "uncertainty" std of kstats, which carries an extra K/(K-1)).  Welford accumulation in fp32 over
 * k = 0..K-1: bitwise repeatable and independent of the other points of the call.  The transcendentals follow the
 * handle's precision as in cfn_flow_composite_fwd.  Arguments are checked before any CUDA call; M == 0 launches nothing.
 * Added without a cfn_version() change: callers detect the feature by the presence of this symbol. */
int cfn_field_stats_f32(const CfnHandle* h, const float* flow_params, const float* eps_alpha, const float* eps_rgb,
                        int64_t M, float* out, void* stream);

/* ---- F7: gradients with respect to the rays and the camera pose (INTEGRATION.md §2) -------------------------------- */
/* Added without a cfn_version() change: callers detect the feature by the presence of these symbols.  Every entry
 * point checks its arguments before any CUDA call.  The calls chain to d loss / d ray_batch for one single-network
 * training-path pass (cfn_network_fwd with save_for_backward + the training flavour of cfn_flow_composite_fwd):
 *   cfn_flow_composite_bwd_rays -> cfn_network_bwd_inputs -> cfn_ray_grad_f32 [-> cfn_rays_from_pose_bwd_f32].
 * A coarse+fine render is two such passes whose g_rays add up.  The coarse pass chains as above.  The fine pass runs on
 * z_all = cfn_merge_sorted_src_f32(coarse z_vals, z_samples) -> (z_all, src), with the resampled depths z_samples
 * (cfn_sample_pdf_f32) held constant, and ends in the merged-grid reduction:
 *   cfn_flow_composite_bwd_rays -> cfn_network_bwd_inputs -> cfn_ray_grad_merged_f32(src, Nc, coarse t_vals / t_rand).
 *
 * cfn_flow_composite_bwd with the same arguments and results, plus two per-sample sums over k (written, not added):
 * g_zdirect (B,N) = sum_k d loss/d depth_map[b,k] * weights[b,n,k] (the depth map's direct z term) and g_delta (B,N) =
 * sum_k d loss / d delta[b,n,k] with delta = dist * |d| the sample distance of raw2outputs (main:427-429).  Both REQUIRED. */
int cfn_flow_composite_bwd_rays(CfnHandle* h, const float* flow_params, const float* z_vals, const float* rays_d,
                                int rays_d_stride, const float* eps_alpha, const float* eps_rgb, int64_t eps_group_rays,
                                int64_t B, int N, int white_bkgd, const float* g_rgb_map, const float* g_depth_map,
                                const float* g_logdet, const float* trans, const float* seg_sums, int n_segments,
                                float* g_flow_params, float* g_globals_partial, float* g_zdirect, float* g_delta,
                                void* stream);

/* Columns of one g_enc row of cfn_network_bwd_inputs: 2 * round8(3 + 6 L_pos) + round8(3 + 6 L_dir) (160 for the
 * canonical network).  0 for a null handle. */
int cfn_input_grad_width(const CfnHandle* h);

/* cfn_network_bwd that also writes the gradients of the encoded network inputs: g_enc (B*N, cfn_input_grad_width), fp32,
 * row m = [d loss/d gamma(p) through layer 0 | through the skip layer (zeros without one) | d loss/d gamma(d) through the
 * view layer], each block padded to a multiple of 8 columns (pad columns are 0).  The two gamma(p) blocks are kept apart
 * (cfn_ray_grad_f32 adds them).  grads may be NULL: then no weight gradient is computed and nothing in grads is touched
 * (a frozen network: about half the backward's dense work); otherwise it is exactly the grads argument of the plain
 * backward. */
int cfn_network_bwd_inputs(CfnHandle* h, const float* g_flow_params, int64_t B, int N, void* workspace,
                           size_t workspace_bytes, float* const* grads, int n_params, float* g_enc, void* stream);

/* g_rays (B,11) = d loss / d rays [o d near far viewdir] from g_enc (cfn_network_bwd_inputs) and g_zdirect / g_delta
 * (cfn_flow_composite_bwd_rays) of the same pass.  rays, t_vals, t_rand, lindisp and z_vals are what cfn_zvals_f32 was
 * given and wrote (t_rand NULL = no stratified jitter; it is data and gets no gradient).  One warp per ray, fixed-order
 * sums: bitwise repeatable. */
int cfn_ray_grad_f32(const CfnHandle* h, const float* rays, const float* z_vals, const float* t_vals, const float* t_rand,
                     int lindisp, const float* g_enc, const float* g_zdirect, const float* g_delta, int64_t B, int N,
                     float* g_rays, void* stream);

/* cfn_ray_grad_f32 for the fine pass of a coarse+fine render: z_vals (B,N) is the merged grid and src (B,N) the
 * permutation cfn_merge_sorted_src_f32 wrote with a = the coarse z_vals (B,Nc), 0 < Nc <= N.  t_vals (Nc), t_rand (B,Nc or
 * NULL) and lindisp are what made the coarse z_vals.  A slot with src < Nc chains its d loss / d z through coarse slot
 * src's schedule (stratified neighbours src -+ 1 of the coarse grid); a slot with src >= Nc is a resampled depth, a
 * constant: it adds nothing to near / far.  o, d and viewdir get the terms of every slot.  Fixed-order sums: bitwise
 * repeatable. */
int cfn_ray_grad_merged_f32(const CfnHandle* h, const float* rays, const float* z_vals, const int32_t* src, int Nc,
                            const float* t_vals, const float* t_rand, int lindisp, const float* g_enc, const float* g_zdirect,
                            const float* g_delta, int64_t B, int N, float* g_rays, void* stream);

/* Adjoint of cfn_rays_from_pose_f32 with the same H, W, focal, ndc, ndc_near: g_rays (H*W,11) -> g_c2w (3,4), the rows
 * of d loss / d c2w[:3,:4] (near / far are constants).  c2w (12 floats) is in DEVICE memory here.  partials: device
 * scratch of CFN_POSE_BWD_PARTIALS floats.  Fixed-order block sums and a fixed-order final pass: bitwise repeatable. */
#define CFN_POSE_BWD_PARTIALS 3072
int cfn_rays_from_pose_bwd_f32(int H, int W, double focal, const float* c2w, int ndc, double ndc_near, const float* g_rays,
                               float* partials, float* g_c2w, void* stream);

/* ---- F3: fused optimiser step (torch.optim.Adam, run_nerf_uncertainty_NF.py:339, 1065-1077) ------------------- */
/* One launch over all n_tensors parameter tensors.  The four pointer arrays and numels live in HOST memory and hold
 * DEVICE pointers / element counts; `step` is the 1-based step count (bias correction), `lr` the already decayed
 * learning rate (main:1073-1077), `grad_scale` multiplies every gradient first (1/world after a sum all-reduce). */
int cfn_adam_step_f32(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                      float* const* exp_avg_sq, const int64_t* numels, float lr, float beta1, float beta2, float eps,
                      int step, float grad_scale, void* stream);

/* Same update with the optimiser clock in DEVICE memory, so that a whole training step can be replayed as one CUDA
 * graph: state_dev (4 floats: step count, learning rate of this step, 1 - beta1^step, sqrt(1 - beta2^step); zero it
 * before the first step) is advanced by one thread and then read by the update kernel.  The learning rate follows the
 * reference's schedule (main:1073-1077, applied after optimizer.step() with a global_step that lags by one):
 * lr(t) = lr0 * decay_rate^(max(t - 2, 0) / decay_steps); decay_steps <= 0 keeps lr0. */
int cfn_adam_step_dev_f32(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                          float* const* exp_avg_sq, const int64_t* numels, float* state_dev, float lr0, float decay_rate,
                          float decay_steps, float beta1, float beta2, float eps, float grad_scale, void* stream);

/* Gradients of the four global latent parameters (models.py:44-48): out8 = sum over rays of g_globals_partial (B,8)
 * (fixed order: deterministic) plus the base log-density part of entropy_coef * loss_entropy
 * (-entropy_coef / alpha_std, -entropy_coef / (3 rgb_std); models.py:268, 283, 286).  out8 = d/d[alpha_mean,
 * alpha_std, rgb_mean(3), rgb_std(3)], i.e. exactly parameter tensors 0..3 when they are stored back to back. */
int cfn_globals_grad_f32(const CfnHandle* h, const float* g_globals_partial, int64_t B, float entropy_coef, float* out8,
                         void* stream);

/* ---- diagnostics ---------------------------------------------------------------------------------- */
/* When CFN_TC_PROFILE=1 is set in the environment at cfn_create time, the tensor-core network kernel records
 * clock64() stamps of CTA 0 (3 roles x 4096: epilogue warp, MMA thread, TMA producer); this copies them to HOST
 * memory after a device synchronise.  Used by scripts/k1_timeline.py only; not part of the data path. */
int cfn_debug_profile(CfnHandle* h, uint64_t* out_host, int n);

/* The dense contraction primitive of the network stage, exposed for unit tests and micro-benchmarks:
 *   C(m,n) = epi( [C(m,n) +] sum_k A[m*a_rs + k*a_cs] * B[k*b_rs + n*b_cs] + bias[n] )      (fp32 storage)
 * engine 0: CUDA-core fp32 FMA (sgemm.cu); engine 1: tcgen05.mma kind::tf32 fed by TMA (gemm_tc.cu; needs unit stride
 * along one axis of each operand and 16-byte aligned bases / strides, else CFN_EINVAL).
 * epilogue: 0 none, 1 ReLU, 2 tanh where aux[n] != 0, 3 zero where aux[m*aux_rs + n] <= 0.  split_k > 1: partial sums
 * are added atomically into a pre-zeroed C (no bias / epilogue).  round_out (engine 1): round outputs to tf32.
 * Replaces the torch.nn.Linear / autograd matmuls of model/models.py:165-186 inside cfn_network_fwd / _bwd. */
int cfn_gemm_f32(int engine, const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs, int64_t b_cs,
                 float* C, int64_t c_rs, const float* bias, const float* aux, int64_t aux_rs, int64_t M, int N, int64_t K,
                 int epilogue, int accumulate, int split_k, int round_out, void* stream);


/* The same primitive with bf16 STORAGE (tensor-core engine only: tcgen05.mma kind::f16, bf16 operands, fp32
 * accumulation): A and B point to bf16 elements (strides in elements, 16-byte aligned bases / strides), C is bf16
 * (c_bf16 = 1) or fp32.  epilogue as above; epilogue 1 can also write relu'(C) as a bit mask (mask_out: one 32-bit word
 * per row and 32 columns, bits_ld words per row; column n at bit 8 * (n % 4) + (n % 32) / 4) and epilogue 3 reads such a mask (aux_bits) instead of an fp32 aux.
 * split_k > 1: fp32 atomics into a pre-zeroed fp32 C; rowsum (optional, pre-zeroed, M floats) += sum_k A(m,k).
 * Instantiated flavours = the ones the training chain issues (else CFN_EINVAL): K-major x K-major {none, ReLU -> bf16;
 * tanh-mask -> fp32}, K-major x N-major {none -> bf16 or fp32 (the input
 * gradients of cfn_network_bwd_inputs), bit-mask -> bf16}, M-major x N-major split-K -> fp32. */
int cfn_gemm_bf16(const void* A, int64_t a_rs, int64_t a_cs, const void* B, int64_t b_rs, int64_t b_cs, void* C,
                  int64_t c_rs, int c_bf16, const float* bias, const float* aux, uint32_t* mask_out,
                  const uint32_t* aux_bits, int64_t bits_ld, int64_t M, int N, int64_t K, int epilogue, int split_k,
                  float* rowsum, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CFNERF_B200_H */
