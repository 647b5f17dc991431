// Per-ray streaming kernels: sample schedule (A1), stand-alone raw2outputs (A8, "K2'"), sample_pdf and
// sorted merge (A9, "K3"), K-mean of weights.  All fp32, HBM-bound, one warp per ray (lane = latent sample k
// or lane = sample along the ray), coalesced 128-bit loads.
#include <math.h>

#include "common.cuh"

namespace cfn {

// ------------------------------------------------------------------------------------------------
// A1: z_vals = near*(1-t) + far*t  (or the lindisp form), optional stratified jitter.
// Reference: run_nerf_uncertainty_NF.py:510-532.  Operation order is reproduced with explicit
// round-to-nearest intrinsics so that no FMA contraction changes the last bit.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float z_of_t(float near, float far, float t, int lindisp) {
  float omt = __fsub_rn(1.0f, t);
  if (!lindisp) return __fadd_rn(__fmul_rn(near, omt), __fmul_rn(far, t));
  float a = __fmul_rn(__fdiv_rn(1.0f, near), omt);
  float b = __fmul_rn(__fdiv_rn(1.0f, far), t);
  return __fdiv_rn(1.0f, __fadd_rn(a, b));
}

__global__ void zvals_kernel(const float* __restrict__ rays, const float* __restrict__ t_vals,
                             const float* __restrict__ t_rand, int lindisp, float* __restrict__ z_vals, int64_t B,
                             int N) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * N) return;
  int64_t b = idx / N;
  int n = (int)(idx - b * N);
  float near = rays[b * 11 + 6], far = rays[b * 11 + 7];
  float z = z_of_t(near, far, t_vals[n], lindisp);
  if (t_rand != nullptr) {
    float upper = z, lower = z;
    if (n < N - 1) upper = __fmul_rn(0.5f, __fadd_rn(z_of_t(near, far, t_vals[n + 1], lindisp), z));
    if (n > 0) lower = __fmul_rn(0.5f, __fadd_rn(z, z_of_t(near, far, t_vals[n - 1], lindisp)));
    z = __fadd_rn(lower, __fmul_rn(__fsub_rn(upper, lower), t_rand[idx]));
  }
  z_vals[idx] = z;
}

int launch_zvals(const float* rays, const float* t_vals, const float* t_rand, int lindisp, float* z_vals, int64_t B,
                 int N, cudaStream_t s) {
  if (B == 0) return CFN_OK;
  int64_t total = B * N;
  zvals_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(rays, t_vals, t_rand, lindisp, z_vals, B, N);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

// ------------------------------------------------------------------------------------------------
// F2: ray generation for a full image (`render(..., c2w=pose)`: run_nerf_uncertainty_NF.py:129-158 with get_rays,
// run_nerf_helpers.py:288-297, and ndc_rays, helpers:360-377).  One thread per pixel writes the (11)-float ray record
// [o d near far viewdir]; the fp32 operation order of the reference expressions is kept with explicit intrinsics.
// ------------------------------------------------------------------------------------------------
struct Pose { float m[12]; };   // c2w[:3,:4] row-major

__global__ void rays_from_pose_kernel(int H, int W, float focal, Pose c2w, float near, float far, int ndc, float ndc_near,
                                      float sW, float sH, float two_near, float* __restrict__ rays) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= H * W) return;
  const int row = p / W, col = p - row * W;
  // dirs = [(i - W/2)/focal, -(j - H/2)/focal, -1]
  const float d0 = __fdiv_rn(__fsub_rn((float)col, (float)W * 0.5f), focal);
  const float d1 = -__fdiv_rn(__fsub_rn((float)row, (float)H * 0.5f), focal);
  const float d2 = -1.0f;
  float dx[3], ox[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {   // rays_d[k] = sum_c dirs[c] * c2w[k][c]
    dx[k] = __fadd_rn(__fadd_rn(__fmul_rn(d0, c2w.m[4 * k + 0]), __fmul_rn(d1, c2w.m[4 * k + 1])), __fmul_rn(d2, c2w.m[4 * k + 2]));
    ox[k] = c2w.m[4 * k + 3];
  }
  // viewdirs are taken BEFORE the NDC warp (main:136-144)
  const float nrm = sqrtf(dx[0] * dx[0] + dx[1] * dx[1] + dx[2] * dx[2]);
  const float v0 = __fdiv_rn(dx[0], nrm), v1 = __fdiv_rn(dx[1], nrm), v2 = __fdiv_rn(dx[2], nrm);
  if (ndc) {
    const float t = __fdiv_rn(-__fadd_rn(ndc_near, ox[2]), dx[2]);
#pragma unroll
    for (int k = 0; k < 3; ++k) ox[k] = __fadd_rn(ox[k], __fmul_rn(t, dx[k]));
    const float o0 = __fdiv_rn(__fmul_rn(sW, ox[0]), ox[2]);
    const float o1 = __fdiv_rn(__fmul_rn(sH, ox[1]), ox[2]);
    const float o2 = __fadd_rn(1.0f, __fdiv_rn(two_near, ox[2]));
    const float e0 = __fmul_rn(sW, __fsub_rn(__fdiv_rn(dx[0], dx[2]), __fdiv_rn(ox[0], ox[2])));
    const float e1 = __fmul_rn(sH, __fsub_rn(__fdiv_rn(dx[1], dx[2]), __fdiv_rn(ox[1], ox[2])));
    const float e2 = __fdiv_rn(-two_near, ox[2]);
    ox[0] = o0; ox[1] = o1; ox[2] = o2;
    dx[0] = e0; dx[1] = e1; dx[2] = e2;
  }
  float* r = rays + (int64_t)p * 11;
  r[0] = ox[0]; r[1] = ox[1]; r[2] = ox[2];
  r[3] = dx[0]; r[4] = dx[1]; r[5] = dx[2];
  r[6] = near; r[7] = far;
  r[8] = v0; r[9] = v1; r[10] = v2;
}

int launch_rays_from_pose(int H, int W, double focal, const float* c2w12, double near, double far, int ndc, double ndc_near,
                          float* rays, cudaStream_t s) {
  CFN_CHECK_ARG(H > 0 && W > 0 && focal > 0 && (int64_t)H * W < (1ll << 31), "rays_from_pose: bad image size");
  Pose pz;
  for (int i = 0; i < 12; ++i) pz.m[i] = c2w12[i];
  // the python scalars of ndc_rays are evaluated in double and rounded once when they meet an fp32 tensor
  const float sW = (float)(-1.0 / ((double)W / (2.0 * focal))), sH = (float)(-1.0 / ((double)H / (2.0 * focal)));
  const float two_near = (float)(2.0 * ndc_near);
  const int n = H * W;
  rays_from_pose_kernel<<<(n + 255) / 256, 256, 0, s>>>(H, W, (float)focal, pz, (float)near, (float)far, ndc, (float)ndc_near,
                                                        sW, sH, two_near, rays);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

// F7: the adjoint of rays_from_pose_kernel.  g_rays (H*W,11) -> g_c2w (3,4) through o = t, d = R dir_cam, the viewdir
// normalisation (taken before the warp) and, with ndc, the NDC warp (helpers:360-377); near / far are constants.  Every
// thread walks a fixed set of pixels, each block joins its 256 threads' 12 sums by a fixed tree, and one final block adds
// the kPoseBwdBlocks partials in order: the result is bitwise repeatable.  c2w is read from device memory.
constexpr int kPoseBwdBlocks = CFN_POSE_BWD_PARTIALS / 12;

__global__ void __launch_bounds__(256)
rays_from_pose_bwd_kernel(int H, int W, float focal, const float* __restrict__ c2w, int ndc, float ndc_near, float sW,
                          float sH, float two_near, const float* __restrict__ g_rays, float* __restrict__ partials) {
  __shared__ float red[12][256];
  float m[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) m[i] = c2w[i];
  float acc[12];
#pragma unroll
  for (int i = 0; i < 12; ++i) acc[i] = 0.f;
  const int n = H * W;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
    const int row = p / W, col = p - row * W;
    const float dir[3] = {__fdiv_rn(__fsub_rn((float)col, (float)W * 0.5f), focal),
                          -__fdiv_rn(__fsub_rn((float)row, (float)H * 0.5f), focal), -1.0f};
    float dx[3];
#pragma unroll
    for (int k = 0; k < 3; ++k)
      dx[k] = __fadd_rn(__fadd_rn(__fmul_rn(dir[0], m[4 * k + 0]), __fmul_rn(dir[1], m[4 * k + 1])), __fmul_rn(dir[2], m[4 * k + 2]));
    const float* g = g_rays + (int64_t)p * 11;
    float go[3] = {g[0], g[1], g[2]}, gd[3] = {g[3], g[4], g[5]};
    // viewdir v = d / |d|:  g_d += (g_v - v (v . g_v)) / |d|
    const float nrm = sqrtf(dx[0] * dx[0] + dx[1] * dx[1] + dx[2] * dx[2]);
    const float v[3] = {dx[0] / nrm, dx[1] / nrm, dx[2] / nrm};
    const float vg = v[0] * g[8] + v[1] * g[9] + v[2] * g[10];
    float gdx[3], gt[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) gdx[k] = (g[8 + k] - v[k] * vg) / nrm;
    if (ndc) {
      // forward: tt = -(near + t_z) / d_z, q = t + tt d, o' = (sW q0/q2, sH q1/q2, 1 + 2n/q2),
      //          d' = (sW (d0/d2 - q0/q2), sH (d1/d2 - q1/q2), -2n/q2)
      const float tt = -(ndc_near + m[11]) / dx[2];
      const float q[3] = {m[3] + tt * dx[0], m[7] + tt * dx[1], m[11] + tt * dx[2]};
      const float iq2 = 1.0f / q[2], iq22 = iq2 * iq2, id2 = 1.0f / dx[2];
      float gq[3];
      gq[0] = (go[0] - gd[0]) * sW * iq2;
      gq[1] = (go[1] - gd[1]) * sH * iq2;
      gq[2] = ((gd[0] - go[0]) * sW * q[0] + (gd[1] - go[1]) * sH * q[1] + (gd[2] - go[2]) * two_near) * iq22;
      float gdd[3];
      gdd[0] = gd[0] * sW * id2;
      gdd[1] = gd[1] * sH * id2;
      gdd[2] = -(gd[0] * sW * dx[0] + gd[1] * sH * dx[1]) * id2 * id2;
      const float gtt = gq[0] * dx[0] + gq[1] * dx[1] + gq[2] * dx[2];
#pragma unroll
      for (int k = 0; k < 3; ++k) { gt[k] = gq[k]; gdx[k] += gdd[k] + gq[k] * tt; }
      // tt = -(near + t_z) / d_z
      gt[2] += -gtt * id2;
      gdx[2] += -gtt * tt * id2;
    } else {
#pragma unroll
      for (int k = 0; k < 3; ++k) { gt[k] = go[k]; gdx[k] += gd[k]; }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
#pragma unroll
      for (int c = 0; c < 3; ++c) acc[4 * k + c] += gdx[k] * dir[c];
      acc[4 * k + 3] += gt[k];
    }
  }
#pragma unroll
  for (int i = 0; i < 12; ++i) red[i][threadIdx.x] = acc[i];
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w)
#pragma unroll
      for (int i = 0; i < 12; ++i) red[i][threadIdx.x] += red[i][threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x < 12) partials[blockIdx.x * 12 + threadIdx.x] = red[threadIdx.x][0];
}

__global__ void pose_bwd_finish_kernel(const float* __restrict__ partials, int n_blocks, float* __restrict__ g_c2w) {
  const int i = threadIdx.x;
  if (i >= 12) return;
  float s = 0.f;
  for (int b = 0; b < n_blocks; ++b) s += partials[b * 12 + i];
  g_c2w[i] = s;
}

int launch_rays_from_pose_bwd(int H, int W, double focal, const float* c2w, int ndc, double ndc_near, const float* g_rays,
                              float* partials, float* g_c2w, cudaStream_t s) {
  CFN_CHECK_ARG(H > 0 && W > 0 && focal > 0 && (int64_t)H * W < (1ll << 31), "rays_from_pose_bwd: bad image size");
  const float sW = (float)(-1.0 / ((double)W / (2.0 * focal))), sH = (float)(-1.0 / ((double)H / (2.0 * focal)));
  const float two_near = (float)(2.0 * ndc_near);
  rays_from_pose_bwd_kernel<<<kPoseBwdBlocks, 256, 0, s>>>(H, W, (float)focal, c2w, ndc, (float)ndc_near, sW, sH, two_near,
                                                          g_rays, partials);
  CFN_LAUNCH_CHECK();
  pose_bwd_finish_kernel<<<1, 32, 0, s>>>(partials, kPoseBwdBlocks, g_c2w);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

// ------------------------------------------------------------------------------------------------
// A8: raw2outputs (run_nerf_uncertainty_NF.py:411-454).  raw (B,N,K,4) is streamed exactly once:
// one warp owns (ray, group of 32 latent samples); lane k walks the N samples front to back carrying the
// transmittance in a register (no scan primitive needed), 512 contiguous bytes per warp per sample.
// Algorithmic traffic: 16NK + 4N + 12 (+4NK with weights) read/written per ray (SURVEY.md §8(d)).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

template <bool WRITE_W>
__global__ void __launch_bounds__(128) raw2outputs_kernel(const float* __restrict__ raw, const float* __restrict__ z_vals,
                                                          const float* __restrict__ rays_d, int rays_d_stride,
                                                          int white_bkgd, float* __restrict__ rgb_map,
                                                          float* __restrict__ disp_map, float* __restrict__ weights,
                                                          float* __restrict__ depth_map, int64_t B, int N, int K,
                                                          int KG) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* sz = smem + warp * 2 * N;
  float* sd = sz + N;
  int64_t wg = (int64_t)blockIdx.x * 4 + warp;
  if (wg >= B * KG) return;
  int64_t b = wg / KG;
  int k = (int)(wg - b * KG) * 32 + lane;
  bool active = k < K;
  for (int n = lane; n < N; n += 32) sz[n] = z_vals[b * N + n];
  const float* d = rays_d + b * rays_d_stride;
  float dx = d[0], dy = d[1], dz = d[2];
  float norm = sqrtf(dx * dx + dy * dy + dz * dz);
  __syncwarp();
  for (int n = lane; n < N; n += 32) sd[n] = ((n < N - 1) ? (sz[n + 1] - sz[n]) : 10.0f) * norm;
  __syncwarp();
  if (!active) return;
  const float4* rp = reinterpret_cast<const float4*>(raw) + (b * N) * K + k;
  float T = 1.0f, cr = 0.f, cg = 0.f, cb = 0.f, depth = 0.f, acc = 0.f;
  float* wp = WRITE_W ? (weights + (b * N) * K + k) : nullptr;
#pragma unroll 8
  for (int n = 0; n < N; ++n) {
    float4 r = ldg_stream(rp + (int64_t)n * K);
    // accurate expf/logf, approximate reciprocal: |error| <= ~1e-7 on every term, well inside the 1e-5 bar, and
    // roughly half the instructions of the log1pf / IEEE-division formulation (the kernel is issue-bound otherwise)
    const float sp = r.w > 20.0f ? r.w : logf(1.0f + expf(r.w));
    float alpha = 1.0f - expf(-sp * sd[n]);
    float w = alpha * T;
    T = T * ((1.0f - alpha) + 1e-10f);
    cr += w * __fdividef(1.0f, 1.0f + expf(-r.x));
    cg += w * __fdividef(1.0f, 1.0f + expf(-r.y));
    cb += w * __fdividef(1.0f, 1.0f + expf(-r.z));
    depth += w * sz[n];
    acc += w;
    if (WRITE_W) wp[(int64_t)n * K] = w;
  }
  float disp = 1.0f / fmaxf(2e-10f, depth / (acc + 1e-10f) + 1e-10f);
  if (white_bkgd) {
    float bg = 1.0f - acc;
    cr += bg; cg += bg; cb += bg;
  }
  rgb_map[(b * 3 + 0) * K + k] = cr;
  rgb_map[(b * 3 + 1) * K + k] = cg;
  rgb_map[(b * 3 + 2) * K + k] = cb;
  disp_map[b * K + k] = disp;
  depth_map[b * K + k] = depth;
}

int launch_raw2outputs(const float* raw, const float* z_vals, const float* rays_d, int rays_d_stride, int white_bkgd,
                       float* rgb_map, float* disp_map, float* weights, float* depth_map, int64_t B, int N, int K,
                       cudaStream_t s) {
  CFN_CHECK_ARG(N >= 2 && N <= 4096 && K >= 1, "raw2outputs: unsupported N=%d K=%d (need 2 <= N <= 4096)", N, K);
  if (B == 0) return CFN_OK;
  int KG = (K + 31) / 32;
  int64_t warps = B * KG;
  unsigned grid = (unsigned)((warps + 3) / 4);
  size_t smem = (size_t)4 * 2 * N * sizeof(float);
  if (weights)
    raw2outputs_kernel<true><<<grid, 128, smem, s>>>(raw, z_vals, rays_d, rays_d_stride, white_bkgd, rgb_map, disp_map,
                                                     weights, depth_map, B, N, K, KG);
  else
    raw2outputs_kernel<false><<<grid, 128, smem, s>>>(raw, z_vals, rays_d, rays_d_stride, white_bkgd, rgb_map,
                                                      disp_map, weights, depth_map, B, N, K, KG);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

// ------------------------------------------------------------------------------------------------
// A9: sample_pdf — bit-exact with oracle/cfnerf_oracle.py::sample_pdf (sequential fp32 sums, IEEE
// division, no FMA contraction).  One warp per ray: lane 0 runs the two sequential scans (the order IS the
// specification), all lanes then invert the CDF for their share of the Nf uniforms by binary search.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) sample_pdf_kernel(const float* __restrict__ bins, const float* __restrict__ weights,
                                                         const float* __restrict__ u, float* __restrict__ samples,
                                                         int32_t* __restrict__ below_out, int64_t B, int M, int Nf) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* cdf = smem + warp * 2 * M;
  float* sb = cdf + M;
  int64_t b = (int64_t)blockIdx.x * 4 + warp;
  if (b >= B) return;
  const float* wrow = weights + b * (M - 1);
  // stage w + 1e-5 into cdf[1..M-1] and the bins
  for (int j = lane; j < M - 1; j += 32) cdf[j + 1] = __fadd_rn(wrow[j], 1e-5f);
  for (int j = lane; j < M; j += 32) sb[j] = bins[b * M + j];
  __syncwarp();
  if (lane == 0) {
    float total = 0.0f;
    for (int j = 1; j < M; ++j) total = __fadd_rn(total, cdf[j]);
    float c = 0.0f;
    cdf[0] = 0.0f;
    for (int j = 1; j < M; ++j) {
      c = __fadd_rn(c, __fdiv_rn(cdf[j], total));
      cdf[j] = c;
    }
  }
  __syncwarp();
  for (int i = lane; i < Nf; i += 32) {
    float uu = u[b * Nf + i];
    // inds = #{j : cdf[j] <= u}  (searchsorted right=True); cdf is non-decreasing
    int lo = 0, hi = M;
    while (lo < hi) {
      int mid = (lo + hi) >> 1;
      if (cdf[mid] <= uu) lo = mid + 1; else hi = mid;
    }
    int below = max(lo - 1, 0), above = min(lo, M - 1);
    float cb = cdf[below], ca = cdf[above];
    float denom = __fsub_rn(ca, cb);
    if (denom < 1e-5f) denom = 1.0f;
    float t = __fdiv_rn(__fsub_rn(uu, cb), denom);
    float bb = sb[below], ba = sb[above];
    samples[b * Nf + i] = __fadd_rn(bb, __fmul_rn(t, __fsub_rn(ba, bb)));
    if (below_out) below_out[b * Nf + i] = below;
  }
}

int launch_sample_pdf(const float* bins, const float* weights, const float* u, float* samples, int32_t* below,
                      int64_t B, int M, int Nf, cudaStream_t s) {
  if (B == 0 || Nf == 0) return CFN_OK;
  CFN_CHECK_ARG(M >= 2 && M <= 2048, "sample_pdf: unsupported M=%d", M);
  unsigned grid = (unsigned)((B + 3) / 4);
  sample_pdf_kernel<<<grid, 128, (size_t)4 * 2 * M * sizeof(float), s>>>(bins, weights, u, samples, below, B, M, Nf);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

// sort(cat[a,b]) per ray by ranking: element i goes to position #{j : v_j < v_i or (v_j == v_i and j < i)}, which is
// torch.sort(stable=True).  SRC also writes src[rank] = i, the index into cat[a,b] of every output slot (the ray
// gradient of a merged grid routes each slot's g_z back through it); src is the last parameter so that the values-only
// flavour keeps its parameter layout.
template <bool SRC>
__global__ void merge_sorted_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out,
                                    int Na, int Nb, int32_t* __restrict__ src) {
  extern __shared__ float v[];
  int64_t ray = blockIdx.x;
  int T = Na + Nb;
  for (int i = threadIdx.x; i < T; i += blockDim.x) v[i] = (i < Na) ? a[ray * Na + i] : b[ray * Nb + (i - Na)];
  __syncthreads();
  for (int i = threadIdx.x; i < T; i += blockDim.x) {
    float x = v[i];
    int rank = 0;
    for (int j = 0; j < T; ++j) {
      float y = v[j];
      rank += (y < x) || (y == x && j < i);
    }
    out[ray * T + rank] = x;
    if (SRC) src[ray * T + rank] = i;
  }
}

int launch_merge_sorted(const float* a, const float* b, float* out, int32_t* src, int64_t B, int Na, int Nb,
                        cudaStream_t s) {
  int T = Na + Nb;
  if (B == 0 || T == 0) return CFN_OK;
  CFN_CHECK_ARG(T >= 1 && T <= 8192, "merge_sorted: unsupported size %d", T);
  int threads = T < 256 ? ((T + 31) / 32) * 32 : 256;
  if (src)
    merge_sorted_kernel<true><<<(unsigned)B, threads, (size_t)T * sizeof(float), s>>>(a, b, out, Na, Nb, src);
  else
    merge_sorted_kernel<false><<<(unsigned)B, threads, (size_t)T * sizeof(float), s>>>(a, b, out, Na, Nb, nullptr);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

__global__ void mean_over_k_kernel(const float* __restrict__ w, float* __restrict__ out, int64_t rows, int K) {
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float s = 0.f;
  for (int k = lane; k < K; k += 32) s += w[row * K + k];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) out[row] = s / (float)K;
}

// ------------------------------------------------------------------------------------------------
// F1: the caller's K-reduction + KDE negative log-likelihood (run_nerf_uncertainty_NF.py:1027-1042) and its
// gradient seed in one pass.  One warp per ray, lanes stride over the K latent samples.
//   mean_k, unbiased std * K/(K-1) (main:1034), bandwidth h = std * (0.8/K)^(-1/7) + 1e-5 (detached, main:1036),
//   p_k = exp(-(x_k - t)^2 / (2 h^2)) * (2 pi)^(-1.5) / h, nll = -log(mean_k p_k + 1e-5).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// one ray's KDE term (warp-wide): returns [sum_c nll_c, sum_c (mean_c - t_c)^2] and writes g (3,K) when g != nullptr
__device__ __forceinline__ void kde_nll_ray(const float* __restrict__ x3, const float* __restrict__ t3, int K, float bw_factor,
                                            float grad_scale, float* __restrict__ g3, int lane, float& nll_sum, float& mse_sum) {
  nll_sum = 0.f; mse_sum = 0.f;
  const float c_norm = 0.06349363593424097f;   // (2*pi)^(-1.5)
  for (int c = 0; c < 3; ++c) {
    const float* x = x3 + c * K;
    const float t = t3[c];
    float s = 0.f;
    for (int k = lane; k < K; k += 32) s += x[k];
    const float m = warp_sum(s) / (float)K;
    float q = 0.f;
    for (int k = lane; k < K; k += 32) { const float dlt = x[k] - m; q += dlt * dlt; }
    const float var = warp_sum(q) / (float)(K - 1);
    const float sd = sqrtf(var) * (float)K / (float)(K - 1);
    const float h = sd * bw_factor + 1e-5f;
    const float inv2h2 = 1.0f / (2.0f * h * h);
    float ps = 0.f;
    for (int k = lane; k < K; k += 32) { const float dlt = x[k] - t; ps += expf(-(dlt * dlt) * inv2h2) * (c_norm / h); }
    const float pm = warp_sum(ps) / (float)K;
    nll_sum += -logf(pm + 1e-5f);
    mse_sum += (m - t) * (m - t);
    if (g3) {
      const float coef = grad_scale / ((pm + 1e-5f) * (float)K * h * h);
      for (int k = lane; k < K; k += 32) {
        const float dlt = x[k] - t;
        g3[c * K + k] = coef * expf(-(dlt * dlt) * inv2h2) * (c_norm / h) * dlt;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// F1, the whole trainer loss of the shipped recipe (colmap_depth, run_nerf_uncertainty_NF.py:1018-1055) in one launch
// over the concatenated batch [B_rgb colour rays | B_depth depth rays] (main:1009-1011); with B_depth = 0 it is the
// plain KDE-NLL loss (api.kde_nll_loss):
//   colour rays: K-mean + KDE-NLL as above (the gradient seed w.r.t. rgb_map; their depth gets no gradient);
//   depth rays : depth = mean_K depth_map (main:1020), squared error against the COLMAP depth (img2mse, main:1053);
//                d/d depth_map[b,k] = depth_scale * 2 * err / K; their colours get no gradient (rgbs[:N_batch], main:1021).
// partial (B,3) = [sum_c nll_c, sum_c (mean_c - t_c)^2, (mean_K depth - target_depth)^2]; the caller takes
// loss_nll = sum(partial[:,0]) / (3 B_rgb), depth_loss = sum(partial[:,2]) / B_depth.
// ------------------------------------------------------------------------------------------------
__global__ void trainer_loss_kernel(const float* __restrict__ rgb_map, const float* __restrict__ depth_map,
                                    const float* __restrict__ target_rgb, const float* __restrict__ target_depth,
                                    int64_t B_rgb, int64_t B_depth, int K, float bw_factor, float nll_scale, float depth_scale,
                                    float* __restrict__ partial, float* __restrict__ g_rgb, float* __restrict__ g_depth) {
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= B_rgb + B_depth) return;
  if (b < B_rgb) {
    float nll_sum, mse_sum;
    kde_nll_ray(rgb_map + b * 3 * K, target_rgb + b * 3, K, bw_factor, nll_scale, g_rgb ? g_rgb + b * 3 * K : nullptr, lane,
                nll_sum, mse_sum);
    if (g_depth) for (int k = lane; k < K; k += 32) g_depth[b * K + k] = 0.f;
    if (lane == 0) { partial[b * 3 + 0] = nll_sum; partial[b * 3 + 1] = mse_sum; partial[b * 3 + 2] = 0.f; }
  } else {
    float s = 0.f;
    for (int k = lane; k < K; k += 32) s += depth_map[b * K + k];
    const float err = warp_sum(s) / (float)K - target_depth[b - B_rgb];
    const float gk = depth_scale * 2.0f * err / (float)K;
    if (g_depth) for (int k = lane; k < K; k += 32) g_depth[b * K + k] = gk;
    if (g_rgb) for (int i = lane; i < 3 * K; i += 32) g_rgb[b * 3 * K + i] = 0.f;
    if (lane == 0) { partial[b * 3 + 0] = 0.f; partial[b * 3 + 1] = 0.f; partial[b * 3 + 2] = err * err; }
  }
}

int launch_trainer_loss(const float* rgb_map, const float* depth_map, const float* target_rgb, const float* target_depth,
                        int64_t B_rgb, int64_t B_depth, int K, float nll_scale, float depth_scale, float* partial, float* g_rgb,
                        float* g_depth, cudaStream_t s) {
  if (B_rgb + B_depth == 0) return CFN_OK;
  CFN_CHECK_ARG(K >= 2, "trainer_loss: K_samples must be >= 2 (unbiased std)");
  const float bw = (float)pow(0.8 / (double)K, -1.0 / 7.0);
  int64_t threads = (B_rgb + B_depth) * 32;
  trainer_loss_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(rgb_map, depth_map, target_rgb, target_depth, B_rgb,
                                                                         B_depth, K, bw, nll_scale, depth_scale, partial, g_rgb,
                                                                         g_depth);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

// gradients of the four global latent parameters (models.py:44-48): the per-ray partial sums of K4 (through
// z0 = eps * std + mean), summed over the rays in a fixed order (deterministic), plus the base log-density of the
// entropy term: -log(std) per latent dimension, i.e. -ent_coef / alpha_std and -ent_coef / (3 rgb_std) (models.py:268,
// 283, 286; the eps^2 part is constant).  out (8) = d/d[alpha_mean, alpha_std, rgb_mean(3), rgb_std(3)].
__global__ void globals_grad_kernel(const float* __restrict__ partial, int64_t B, const float* __restrict__ globals8,
                                    float ent_coef, float* __restrict__ out) {
  __shared__ float red[8][8];
  const int j = threadIdx.x & 7, part = threadIdx.x >> 3;   // 64 threads: 8 columns x 8 row slices
  float s = 0.f;
  for (int64_t b = part; b < B; b += 8) s += partial[b * 8 + j];
  red[part][j] = s;
  __syncthreads();
  if (threadIdx.x < 8) {
    float t = 0.f;
#pragma unroll
    for (int p = 0; p < 8; ++p) t += red[p][j];
    if (j == 1) t -= ent_coef / globals8[1];
    if (j >= 5) t -= ent_coef / (3.0f * globals8[j]);
    out[j] = t;
  }
}

int launch_globals_grad(const float* partial, int64_t B, const float* globals8, float ent_coef, float* out, cudaStream_t s) {
  globals_grad_kernel<<<1, 64, 0, s>>>(partial, B, globals8, ent_coef, out);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

int launch_mean_over_k(const float* w, float* out, int64_t rows, int K, cudaStream_t s) {
  if (rows == 0) return CFN_OK;
  int64_t threads = rows * 32;
  mean_over_k_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(w, out, rows, K);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

}  // namespace cfn
