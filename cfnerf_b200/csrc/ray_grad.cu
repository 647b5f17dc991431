// F7: gradients with respect to the ray record.  The encoding backward and the per-ray reduction that turn the input
// gradients of the network chain (chain_network_bwd's g_enc) and K4's per-sample sums (the RAYGRAD flavour: g_zdirect,
// g_delta) into g_rays (B,11) = d L / d [o d near far viewdir]  (SURVEY Appendix A.2 for the compositing terms):
//   g_p_n   = g_gamma(p)[x] + sum_l 2^l (cos(2^l p) g_sin_l - sin(2^l p) g_cos_l)          (per point, both gamma(p) blocks)
//   g_z_n   = d . g_p_n + g_zdirect_n + |d| (g_delta_{n-1} - g_delta_n)                     (delta_n = (z_{n+1} - z_n) |d|)
//   g_o     = sum_n g_p_n
//   g_d     = sum_n z_n g_p_n + (sum_n g_delta_n dist_n) d / |d|                            (dist_{N-1} = 10)
//   near/far: g_z_n through zvals_kernel's schedule (linear or lindisp; the stratified mids / lower / upper when t_rand is
//             given; t_rand itself is data); on a merged coarse+fine grid only the slots taken from the coarse grid,
//             through the coarse schedule (the MERGED flavour)
//   viewdir: J_gamma(vd)^T sum_n g_gamma(d)_n                                              (vd is constant along a ray)
// One warp per ray, lane = sample; every sum runs in a fixed order (lane-sequential, then a fixed xor butterfly), so the
// result is bitwise repeatable.  The points are recomputed in the forward encoder's fp32 operation order and the
// encoding is differentiated with the accurate sincosf, as the forward encoder evaluates it (frequencies reach 2^9).
#include <math.h>

#include "common.cuh"

namespace cfn {

constexpr int kRayGradMaxDir = 104;   // 3 + 6 * 16 view-encoding columns (+ pad)

__device__ __forceinline__ float zsched(float near, float far, float t, int lindisp) {
  const float omt = __fsub_rn(1.0f, t);
  if (!lindisp) return __fadd_rn(__fmul_rn(near, omt), __fmul_rn(far, t));
  return __fdiv_rn(1.0f, __fadd_rn(__fmul_rn(__fdiv_rn(1.0f, near), omt), __fmul_rn(__fdiv_rn(1.0f, far), t)));
}

// (d z / d near, d z / d far) of the unperturbed schedule at t
__device__ __forceinline__ void zsched_grad(float near, float far, float t, int lindisp, float& cn, float& cf) {
  if (!lindisp) { cn = 1.0f - t; cf = t; return; }
  const float z = zsched(near, far, t, lindisp), zz = z * z;
  cn = zz * (1.0f - t) / (near * near);
  cf = zz * t / (far * far);
}

// MERGED: z_vals is a merged grid (the fine pass of a coarse+fine render) whose slot n holds element src[b,n] of
// cat[coarse z (Nc), resampled z]; t_vals (Nc) and t_rand (B,Nc) are the coarse pass's.  A slot taken from the coarse
// grid chains its g_z through coarse slot src's schedule (stratified neighbours src -+ 1 of the coarse grid); a
// resampled slot is a constant (sample_pdf is not differentiated) and adds nothing to near / far.  src and Nc come last
// so that the plain flavour keeps its parameter layout.
template <bool MERGED>
__global__ void __launch_bounds__(128)
ray_grad_kernel(const float* __restrict__ rays, const float* __restrict__ z_vals, const float* __restrict__ t_vals,
                const float* __restrict__ t_rand, int lindisp, const float* __restrict__ g_enc, int ld_enc, int gp,
                int has_skip, int L_pos, int L_dir, const float* __restrict__ g_zdirect, const float* __restrict__ g_delta,
                int64_t B, int N, float* __restrict__ g_rays, const int32_t* __restrict__ src, int Nc) {
  __shared__ float s_gd[4][kRayGradMaxDir];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b = (int64_t)blockIdx.x * 4 + warp;
  if (b >= B) return;
  const float* r = rays + b * 11;
  const float o[3] = {r[0], r[1], r[2]};
  const float d[3] = {r[3], r[4], r[5]};
  const float near = r[6], far = r[7];
  const float norm = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
  const float* zr = z_vals + b * N;
  const float* gzd = g_zdirect + b * N;
  const float* gdl = g_delta + b * N;
  float acc[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // g_o (3) | sum z g_p (3) | sum g_delta dist | near | far
  for (int n = lane; n < N; n += 32) {
    const float z = zr[n];
    const float* row = g_enc + (b * N + n) * ld_enc;
    const float* row2 = row + gp;
    float gpt[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float p = __fadd_rn(o[c], __fmul_rn(d[c], z));   // main:534, as the forward encoder evaluates it
      float g = row[c] + (has_skip ? row2[c] : 0.f);
      float f = 1.0f;
      for (int l = 0; l < L_pos; ++l) {
        const int i = 3 + 6 * l + c;
        const float gs = row[i] + (has_skip ? row2[i] : 0.f);
        const float gc = row[i + 3] + (has_skip ? row2[i + 3] : 0.f);
        float sn, cs;
        sincosf(p * f, &sn, &cs);
        g += f * (cs * gs - sn * gc);
        f *= 2.0f;
      }
      gpt[c] = g;
    }
    const float dl = gdl[n];
    float gz = d[0] * gpt[0] + d[1] * gpt[1] + d[2] * gpt[2] + gzd[n];
    gz += norm * ((n > 0 ? gdl[n - 1] : 0.f) - (n < N - 1 ? dl : 0.f));
    const float dist = (n < N - 1) ? (zr[n + 1] - z) : 10.0f;
#pragma unroll
    for (int c = 0; c < 3; ++c) { acc[c] += gpt[c]; acc[3 + c] += z * gpt[c]; }
    acc[6] += dl * dist;
    // z_n through the schedule: lower + (upper - lower) * t_rand with lower / upper the neighbouring mids; on a merged
    // grid the schedule slot is the coarse slot m the sample came from (Ns = Nc slots)
    const int m = MERGED ? src[b * N + n] : n;
    const int Ns = MERGED ? Nc : N;
    if (!MERGED || m < Nc) {
      float cn, cf;
      zsched_grad(near, far, t_vals[m], lindisp, cn, cf);
      if (t_rand) {
        float pn = cn, pf = cf, qn = cn, qf = cf;   // d lower, d upper
        if (m > 0) { float an, af; zsched_grad(near, far, t_vals[m - 1], lindisp, an, af); pn = 0.5f * (cn + an); pf = 0.5f * (cf + af); }
        if (m < Ns - 1) { float an, af; zsched_grad(near, far, t_vals[m + 1], lindisp, an, af); qn = 0.5f * (an + cn); qf = 0.5f * (af + cf); }
        const float u = t_rand[b * Ns + m];
        cn = pn + (qn - pn) * u;
        cf = pf + (qf - pf) * u;
      }
      acc[7] += gz * cn;
      acc[8] += gz * cf;
    }
  }
#pragma unroll
  for (int j = 0; j < 9; ++j)
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], s);
  // sum of g_gamma(d) over the samples, lane = encoding column
  const int in_dir = 3 + 6 * L_dir;
  const float* gdir = g_enc + (b * N) * ld_enc + 2 * gp;
  for (int j = lane; j < in_dir; j += 32) {
    float sum = 0.f;
    for (int n = 0; n < N; ++n) sum += gdir[(int64_t)n * ld_enc + j];
    s_gd[warp][j] = sum;
  }
  __syncwarp();
  float* out = g_rays + b * 11;
  if (lane < 3) {
    const int c = lane;
    const float vd = r[8 + c];
    float g = s_gd[warp][c];
    float f = 1.0f;
    for (int l = 0; l < L_dir; ++l) {
      float sn, cs;
      sincosf(vd * f, &sn, &cs);
      g += f * (cs * s_gd[warp][3 + 6 * l + c] - sn * s_gd[warp][6 + 6 * l + c]);
      f *= 2.0f;
    }
    out[8 + c] = g;
  }
  if (lane == 0) {
    const float sd = acc[6] / norm;
#pragma unroll
    for (int c = 0; c < 3; ++c) { out[c] = acc[c]; out[3 + c] = acc[3 + c] + sd * d[c]; }
    out[6] = acc[7];
    out[7] = acc[8];
  }
}

int launch_ray_grad(const float* rays, const float* z_vals, const float* t_vals, const float* t_rand, int lindisp,
                    const float* g_enc, int ld_enc, int gp, int has_skip, int L_pos, int L_dir, const float* g_zdirect,
                    const float* g_delta, int64_t B, int N, float* g_rays, cudaStream_t s, const int32_t* src, int Nc) {
  if (B == 0) return CFN_OK;
  CFN_CHECK_ARG(3 + 6 * L_dir <= kRayGradMaxDir, "ray_grad: multires_views %d unsupported", L_dir);
  const unsigned grid = (unsigned)((B + 3) / 4);
  if (src)
    ray_grad_kernel<true><<<grid, 128, 0, s>>>(rays, z_vals, t_vals, t_rand, lindisp, g_enc, ld_enc, gp, has_skip, L_pos,
                                               L_dir, g_zdirect, g_delta, B, N, g_rays, src, Nc);
  else
    ray_grad_kernel<false><<<grid, 128, 0, s>>>(rays, z_vals, t_vals, t_rand, lindisp, g_enc, ld_enc, gp, has_skip, L_pos,
                                                L_dir, g_zdirect, g_delta, B, N, g_rays, nullptr, 0);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

}  // namespace cfn
