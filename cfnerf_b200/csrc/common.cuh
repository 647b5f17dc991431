// Shared declarations of the cfnerf_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/cfnerf_b200.h"

namespace cfn {

void set_error(const char* fmt, ...);

#define CFN_CHECK_ARG(cond, ...)          \
  do {                                    \
    if (!(cond)) {                        \
      ::cfn::set_error(__VA_ARGS__);      \
      return CFN_EINVAL;                  \
    }                                     \
  } while (0)

#define CFN_CUDA(expr)                                                                        \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      ::cfn::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return CFN_ECUDA;                                                                       \
    }                                                                                         \
  } while (0)

#define CFN_LAUNCH_CHECK() CFN_CUDA(cudaGetLastError())

// ---- per-device process state ---------------------------------------------------------------------------
// cudaFuncSetAttribute and the SM count belong to ONE device; an Engine may be created on any device of the process
// (and from any thread), so "done once" flags are kept per device ordinal.  Setting an attribute twice is harmless,
// which makes the relaxed atomics sufficient.
constexpr int kMaxDevices = 64;
inline int current_device() { int d = 0; cudaGetDevice(&d); return (d >= 0 && d < kMaxDevices) ? d : 0; }
struct PerDeviceOnce {
  std::atomic<unsigned long long> mask{0};
  bool done() const { return (mask.load(std::memory_order_acquire) >> current_device()) & 1ull; }
  void mark() { mask.fetch_or(1ull << current_device(), std::memory_order_release); }
};
inline int device_num_sms() {
  static std::atomic<int> n[kMaxDevices];
  const int d = current_device();
  int v = n[d].load(std::memory_order_relaxed);
  if (v <= 0) {
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, d);
    if (v <= 0) v = 148;
    n[d].store(v, std::memory_order_relaxed);
  }
  return v;
}

// ---- fp32 math of the non-GEMM kernels (the library is compiled WITHOUT --use_fast_math) --------------
// Two flavours.  FAST = false: accurate libdevice functions, used by the fp32 "check" path (1e-5 bar).
// FAST = true: one MUFU exp / log / reciprocal per transcendental (absolute error <= ~3e-7 on the bounded outputs
// sigmoid / tanh / alpha), used behind the bf16 / fp16 tensor-core network stage whose bar is 2e-3: the streaming
// kernels are instruction-bound on these functions, not HBM-bound.
template <bool FAST> __device__ __forceinline__ float exp_(float x) { return FAST ? __expf(x) : expf(x); }
template <bool FAST> __device__ __forceinline__ float sigmoid_(float x) {
  return FAST ? __fdividef(1.0f, 1.0f + __expf(-x)) : 1.0f / (1.0f + expf(-x));
}
// F.softplus(beta=1, threshold=20) (run_nerf_uncertainty_NF.py:424)
template <bool FAST> __device__ __forceinline__ float softplus_(float x) {
  if (FAST) return x > 20.0f ? x : __logf(1.0f + __expf(x));
  return x > 20.0f ? x : log1pf(expf(x));
}
// log of the log-det terms (arguments in (1e-8, ~2]): one MUFU.LG2 in the fast flavour (absolute error ~2e-7)
template <bool FAST> __device__ __forceinline__ float log_(float x) { return FAST ? __logf(x) : logf(x); }
template <bool FAST> __device__ __forceinline__ float tanh_(float x) {
  if (FAST) { const float t = __expf(2.0f * x); return 1.0f - __fdividef(2.0f, t + 1.0f); }
  return tanhf(x);
}
__device__ __forceinline__ float sigmoidf_(float x) { return sigmoid_<false>(x); }
__device__ __forceinline__ float softplusf_(float x) { return softplus_<false>(x); }

// flow-parameter record per 3-D point: [alpha d1[F] | alpha d2[F] | alpha b[F] | rgb flow 0 (15) | ... ]
// rgb flow f (15): R1_00 R1_01 R1_02 R1_11 R1_12 R1_22 | R2_00 R2_01 R2_02 R2_11 R2_12 R2_22 | b0 b1 b2
constexpr int kRgbFlowRec = 15;
__host__ __device__ inline int flow_param_width(int F) { return 18 * F; }

// ---- kernels implemented across the .cu files ----------------------------------------------------
int launch_zvals(const float* rays, const float* t_vals, const float* t_rand, int lindisp, float* z_vals, int64_t B,
                 int N, cudaStream_t s);
int launch_rays_from_pose(int H, int W, double focal, const float* c2w12, double near, double far, int ndc, double ndc_near,
                          float* rays, cudaStream_t s);
int launch_raw2outputs(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride, int white_bkgd,
                       float* rgb_map, float* disp_map, float* weights, float* depth_map, int64_t B, int N, int K,
                       cudaStream_t s);
int launch_sample_pdf(const float* bins, const float* weights, const float* u, float* samples, int32_t* below,
                      int64_t B, int M, int Nf, cudaStream_t s);
int launch_merge_sorted(const float* a, const float* b, float* out, int32_t* src, int64_t B, int Na, int Nb,
                        cudaStream_t s);
int launch_trainer_loss(const float* rgb_map, const float* depth_map, const float* target_rgb, const float* target_depth,
                        int64_t B_rgb, int64_t B_depth, int K, float nll_scale, float depth_scale, float* partial, float* g_rgb,
                        float* g_depth, cudaStream_t s);
int launch_adam(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                float* const* exp_avg_sq, const int64_t* numels, float lr, float beta1, float beta2, float eps, int step,
                float grad_scale, cudaStream_t s);
int launch_adam_dev(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                    float* const* exp_avg_sq, const int64_t* numels, float* state, float lr0, float decay_rate,
                    float decay_steps, float beta1, float beta2, float eps, float grad_scale, cudaStream_t s);
int launch_globals_grad(const float* partial, int64_t B, const float* globals8, float ent_coef, float* out, cudaStream_t s);
int launch_mean_over_k(const float* w, float* out, int64_t rows, int K, cudaStream_t s);
int launch_eval_records(const float* kstats, const float* partial, const float* target_rgb, const float* depth_map,
                        const float* target_depth, int64_t B, int K, float* u, float* sq_err, float* abs_err, float* nll,
                        float* depth_u, float* depth_sq_err, float* depth_abs_err, cudaStream_t s);
int sparsify_workspace_bytes(int64_t V, int64_t P, int S, size_t* out);
int launch_sparsify(const float* u, const float* e, const float* a, int64_t V, int64_t P, int S, void* workspace,
                    size_t workspace_bytes, float* curves, float* ause, cudaStream_t s);
int launch_field_stats(int fast_math, int F, int K, const float* globals, const float* flow_params, const float* eps_alpha,
                       const float* eps_rgb, int64_t M, float* out, cudaStream_t s);

int launch_ray_grad(const float* rays, const float* z_vals, const float* t_vals, const float* t_rand, int lindisp,
                    const float* g_enc, int ld_enc, int gp, int has_skip, int L_pos, int L_dir, const float* g_zdirect,
                    const float* g_delta, int64_t B, int N, float* g_rays, cudaStream_t s,
                    const int32_t* src = nullptr, int Nc = 0);
int launch_rays_from_pose_bwd(int H, int W, double focal, const float* c2w, int ndc, double ndc_near, const float* g_rays,
                              float* partials, float* g_c2w, cudaStream_t s);

int launch_flow_composite_fwd(int fast_math, int F, int K, const float* globals, const float* flow_params, const float* z_vals,
                              const float* rays_d, int rays_d_stride, const float* eps_alpha, const float* eps_rgb,
                              int64_t eps_group_rays, int64_t B, int N, int white_bkgd, float* rgb_map, float* disp_map,
                              float* depth_map, float* raw, float* weights, float* logdet_sums, float* kstats, float* trans,
                              float* seg_sums, int n_seg, cudaStream_t s);
int launch_flow_composite_bwd(int fast_math, int F, int K, const float* globals, const float* flow_params, const float* z_vals,
                              const float* rays_d, int rays_d_stride, const float* eps_alpha, const float* eps_rgb,
                              int64_t eps_group_rays, int64_t B, int N, int white_bkgd, const float* g_rgb_map,
                              const float* g_depth_map, const float* g_ld, const float* trans, const float* seg_sums,
                              int n_seg, float* g_flow_params, float* g_globals, cudaStream_t s,
                              float* g_zdirect = nullptr, float* g_delta = nullptr);   // both or neither: ray flavour

// C[m,n] = epi( sum_k A(m,k) * B(k,n) + bias[n] ) with arbitrary element strides (fp32 CUDA-core GEMM).
enum Epilogue { EPI_NONE = 0, EPI_RELU = 1, EPI_TANH_MASK = 2, EPI_RELU_MASK_MUL = 3 };
struct GemmArgs {
  const float* A; int64_t a_rs, a_cs;   // A(m,k) = A[m*a_rs + k*a_cs]
  const float* B; int64_t b_rs, b_cs;   // B(k,n) = B[k*b_rs + n*b_cs]
  float* C; int64_t c_rs;               // C(m,n) = C[m*c_rs + n]
  const float* bias;                    // (N) or nullptr
  const float* aux; int64_t aux_rs;     // EPI_TANH_MASK: aux = per-column flag (N); EPI_RELU_MASK_MUL: aux(m,n) activation, C *= (aux>0)
  int64_t M; int N; int64_t K;
  int epilogue;
  int accumulate;                       // C += result (applied before the epilogue)
  int split_k;                          // >1: atomicAdd partial sums into a pre-zeroed C (no bias/epilogue)
  float* rowsum;                        // tensor-core engine, split_k > 1 only: rowsum[m] += sum_k A(m,k) (pre-zeroed; the bias
                                        // gradient of a wgrad, produced by one extra N=16 MMA against a tile of ones)
  // tensor-core engine only: ReLU derivative as a bit mask, one word per row and 32 output columns (bits_ld words/row;
  // column n of the chunk sits at bit 8 * (n % 4) + (n % 32) / 4 — the order the epilogue's warp votes produce).
  // EPI_RELU writes it (mask_out); EPI_RELU_MASK_MUL reads it (aux_bits) instead of the fp32 aux, 32x fewer bytes.
  uint32_t* mask_out;
  const uint32_t* aux_bits;
  int64_t bits_ld;
  // tensor-core engine only: bf16 STORAGE.  ab_bf16: A and B point to __nv_bfloat16 (strides in elements, tcgen05
  // kind::f16 with bf16 operands); c_bf16: C is written as bf16 (else fp32).  Accumulation is fp32 either way.
  int ab_bf16, c_bf16;
  // split_k > 1 only, opt-in determinism: instead of fp32 atomics into C every split stores its partial product as a
  // dense (M x N) slab in `partials` (capacity partials_floats; the row sums follow the slabs) and a second pass adds the
  // slabs in split order — bitwise run-to-run stable weight gradients (SURVEY 7.3-5).  C need not be pre-zeroed then.
  float* partials; int64_t partials_floats;
};
// C(m,n) = sum_z partials[z][m][n] (fixed order), rowsum_out[m] = sum_z rowsum_partials[z][m] when given
int reduce_split_partials(const float* partials, int split, int64_t M, int N, float* C, int64_t c_rs,
                          const float* rowsum_partials, float* rowsum_out, cudaStream_t s);
int launch_sgemm(const GemmArgs& g, cudaStream_t s);
// same contract on the tensor cores (tcgen05.mma kind::tf32, TMA-fed; gemm_tc.cu).  round_out: round the stored
// outputs to the tf32 grid (they are the next GEMM's operands).
bool tgemm_supported(const GemmArgs& g);
int launch_tgemm(const GemmArgs& g, int round_out, cudaStream_t s);
// true when launch_tgemm can also produce g.rowsum (every CTA (pair) owns exactly one K slice of one tile)
bool tgemm_can_rowsum(const GemmArgs& g);

}  // namespace cfn
