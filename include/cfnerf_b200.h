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
 * reads instead of recomputing it; optional seg_sums (B, n_segments, 5, K) (training flavour only; N must be a multiple
 * of n_segments): per equal sample range of every ray the sums of w*rgb (3), w*z and w — they let the backward walk the
 * n_segments ranges of a ray in independent warps.  Any optional pointer may be NULL. */
int cfn_flow_composite_fwd(CfnHandle* h, const float* flow_params, const float* z_vals, const float* rays_d,
                           int rays_d_stride, const float* eps_alpha, const float* eps_rgb, int64_t eps_group_rays,
                           int64_t B, int N, int white_bkgd, float* rgb_map, float* disp_map, float* depth_map,
                           float* raw, float* weights, float* logdet_sums, float* kstats, float* trans, float* seg_sums,
                           int n_segments, void* stream);

/* Backward (SURVEY.md Appendix A).  g_rgb_map (B,3,K) and g_depth_map (B,K) (NULL = zero) are upstream
 * gradients; g_logdet_alpha / g_logdet_rgb are d loss / d(sum of log-dets) (scalars, e.g. -beta1/(B*N*K)).
 * trans (B,N,K) is REQUIRED device memory: with trans_valid != 0 it holds what cfn_flow_composite_fwd wrote for the
 * same inputs; with trans_valid == 0 it is scratch that this call fills first (an alpha-stack-only pre-pass).
 * seg_sums / n_segments: what cfn_flow_composite_fwd wrote for the same inputs (NULL / 1: one warp walks the whole ray;
 * n_segments > 1 gives small batches n_segments times the parallelism — the reference trains on 512 rays per step).
 * Writes g_flow_params (B*N,18F) and g_globals_partial (B*n_segments,8): per ray and range the
 * partial sums of d/d[alpha_mean, alpha_std, rgb_mean(3), rgb_std(3)] through z0 = eps*std+mean only (the caller sums
 * the rows; kept apart so the result is deterministic). */
int cfn_flow_composite_bwd(CfnHandle* h, const float* flow_params, const float* z_vals, const float* rays_d,
                           int rays_d_stride, const float* eps_alpha, const float* eps_rgb, int64_t eps_group_rays,
                           int64_t B, int N, int white_bkgd, const float* g_rgb_map, const float* g_depth_map,
                           float g_logdet_alpha, float g_logdet_rgb, float* trans, int trans_valid,
                           const float* seg_sums, int n_segments, float* g_flow_params, float* g_globals_partial,
                           void* stream);
/* Same, with PER-RAY log-det gradient seeds read from DEVICE memory: g_logdet_dev (B,2), [b][0] = alpha, [b][1] = rgb.
 * The host does not have to wait for the loss graph before it issues the backward (no device-to-host sync per step),
 * and rays of different network calls / loss terms can carry different seeds (the depth rays of the shipped recipe
 * take no part in the entropy term, main:1018-1023, 1045). */
int cfn_flow_composite_bwd_dev(CfnHandle* h, const float* flow_params, const float* z_vals, const float* rays_d,
                               int rays_d_stride, const float* eps_alpha, const float* eps_rgb, int64_t eps_group_rays,
                               int64_t B, int N, int white_bkgd, const float* g_rgb_map, const float* g_depth_map,
                               const float* g_logdet_dev, float* trans, int trans_valid, const float* seg_sums,
                               int n_segments, float* g_flow_params, float* g_globals_partial, void* stream);

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
/* mean over K of weights (B,N,K) -> (B,N)  (the shared fine grid decision, SURVEY.md A9) */
int cfn_mean_over_k_f32(const float* w, float* out, int64_t rows, int K, void* stream);

/* ---- F1: K-reduction + KDE negative log-likelihood of the trainer (run_nerf_uncertainty_NF.py:1027-1042) ------ */
/* rgb_map (B,3,K), target (B,3) -> partial (B,2) = per-ray [sum_c nll_c, sum_c (mean_k rgb - target)^2] and, when
 * g_rgb_map != NULL, g_rgb_map (B,3,K) = grad_scale * d(sum_c nll_c)/d rgb_map (bandwidth detached as in main:1036).
 * The trainer's loss_nll is sum(partial[:,0]) / (3B); pass grad_scale = 1/(3B) to get its gradient directly. */
int cfn_kde_nll_f32(const float* rgb_map, const float* target, int64_t B, int K, float grad_scale, float* partial,
                    float* g_rgb_map, void* stream);

/* The whole loss of the shipped recipe (--colmap_depth, --depth_lambda; run_nerf_uncertainty_NF.py:1018-1055) over the
 * concatenated batch [B_rgb colour rays | B_depth depth rays] (main:1009-1011) in one launch.  rgb_map (B,3,K),
 * depth_map (B,K) with B = B_rgb + B_depth; target_rgb (B_rgb,3); target_depth (B_depth) (may be NULL when B_depth = 0).
 * partial (B,3) = per-ray [sum_c nll_c, sum_c (mean_k rgb - target)^2, (mean_k depth - target_depth)^2] (colour rays fill
 * columns 0-1, depth rays column 2).  g_rgb_map (B,3,K) = nll_scale * d(sum_c nll_c)/d rgb_map on colour rays, 0 on
 * depth rays (rgbs[:N_batch], main:1021); g_depth_map (B,K) = depth_scale * d(err^2)/d depth_map on depth rays, 0 on
 * colour rays.  Pass nll_scale = 1/(3 B_rgb) and depth_scale = depth_lambda / B_depth to seed the backward directly. */
int cfn_trainer_loss_f32(const float* rgb_map, const float* depth_map, const float* target_rgb, const float* target_depth,
                         int64_t B_rgb, int64_t B_depth, int K, float nll_scale, float depth_scale, float* partial,
                         float* g_rgb_map, float* g_depth_map, void* stream);

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
 * tanh-mask -> fp32}, K-major x N-major {none, bit-mask -> bf16}, M-major x N-major split-K -> fp32. */
int cfn_gemm_bf16(const void* A, int64_t a_rs, int64_t a_cs, const void* B, int64_t b_rs, int64_t b_cs, void* C,
                  int64_t c_rs, int c_bf16, const float* bias, const float* aux, uint32_t* mask_out,
                  const uint32_t* aux_bits, int64_t bits_ld, int64_t M, int N, int64_t K, int epilogue, int split_k,
                  float* rowsum, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CFNERF_B200_H */
