// F6 field-space statistics: for every query point, the mean and the sample std over the K latent draws of the density
// sigma_k = softplus(za_k) (run_nerf_uncertainty_NF.py:424) and of the colour c_k = sigmoid(z_k) (main:431), written as
// (M,8) [sigma mean, sigma std, rgb mean (3), rgb std (3)].  std = sqrt(sum_k (x_k - mean)^2 / (K - 1)), 0 when K = 1:
// the plain sample std, not the "uncertainty" std of kstats (that one carries the reference's extra K/(K-1), main:1034).
//
// Layout: one thread per point, looping over k.  A block of kFieldThreads points stages its (kFieldThreads, 18F) flow
// records (written by K1) through shared memory with coalesced loads, at an odd row stride (18F + 1) so that the
// per-thread row reads are free of bank conflicts; the K base latents z0 = eps * std + mean are computed once per block
// and read back as shared-memory broadcasts.  No cross-lane reduction, no idle lane for K < 32, one code path for
// K = 1..1024.  Each point accumulates with Welford's update in fp32 in the order k = 0, 1, ..., K-1, so the result is
// bitwise repeatable and independent of which other points share the launch.
#include "common.cuh"

namespace cfn {

namespace {

constexpr int kFieldThreads = 128;

// Welford's update of (mean, m2) with the sample x; inv = 1 / (number of samples so far, x included)
__device__ __forceinline__ void welford(float x, float inv, float& mean, float& m2) {
  const float d = x - mean;
  mean += d * inv;
  m2 += d * (x - mean);
}

}  // namespace

template <bool FAST, int FT>
__global__ void __launch_bounds__(kFieldThreads)
field_stats_kernel(int F_rt, int K, const float* __restrict__ globals, const float* __restrict__ flow_params,
                   const float* __restrict__ eps_alpha, const float* __restrict__ eps_rgb, int64_t M,
                   float* __restrict__ out) {
  extern __shared__ __align__(16) float smem[];
  const int F = FT > 0 ? FT : F_rt;
  const int PP = 18 * F;
  const int ld = PP + 1;                                   // odd row stride: conflict-free per-thread row reads
  float4* sz0 = reinterpret_cast<float4*>(smem);           // (K) base latents [rgb 0, 1, 2 | alpha]
  float* sinv = smem + 4 * K;                              // (K) 1 / (k + 1)
  float* srec = sinv + K;                                  // (kFieldThreads, ld) flow records of the block
  const int t = threadIdx.x;
  const int64_t p0 = (int64_t)blockIdx.x * kFieldThreads;
  const int np = (int)min((int64_t)kFieldThreads, M - p0);

  // z0 = eps * std + mean (models.py:200/206), the expressions of flow_composite.cu:99-100
  const float a_mean = globals[0], a_std = globals[1];
  const float c_mean0 = globals[2], c_mean1 = globals[3], c_mean2 = globals[4];
  const float c_std0 = globals[5], c_std1 = globals[6], c_std2 = globals[7];
  for (int k = t; k < K; k += kFieldThreads) {
    const float ea = eps_alpha[k];
    const float e0 = eps_rgb[k * 3 + 0], e1 = eps_rgb[k * 3 + 1], e2 = eps_rgb[k * 3 + 2];
    sz0[k] = make_float4(e0 * c_std0 + c_mean0, e1 * c_std1 + c_mean1, e2 * c_std2 + c_mean2, ea * a_std + a_mean);
    sinv[k] = 1.0f / (float)(k + 1);
  }
  // the block's records are contiguous in global memory: consecutive threads read consecutive floats
  const float* src = flow_params + p0 * PP;
  for (int i = t; i < np * PP; i += kFieldThreads) {
    const int r = i / PP;
    srec[r * ld + (i - r * PP)] = src[i];
  }
  __syncthreads();
  if (t >= np) return;

  const float* P = srec + t * ld;
  float rec[FT > 0 ? 18 * FT : 1];
  if (FT > 0) {
#pragma unroll
    for (int j = 0; j < 18 * FT; ++j) rec[j] = P[j];
    P = rec;
  }

  float s_mean = 0.f, s_m2 = 0.f;
  float r_mean = 0.f, r_m2 = 0.f, g_mean = 0.f, g_m2 = 0.f, b_mean = 0.f, b_m2 = 0.f;
  for (int k = 0; k < K; ++k) {
    const float4 z0 = sz0[k];
    // ---- alpha stack (z_size 1; the flip is the identity): flow_composite.cu:140-148 ----
    float za = z0.w;
#pragma unroll
    for (int f = 0; f < F; ++f) {
      const float d1 = P[f], d2 = P[F + f], bb = P[2 * F + f];
      const float th = tanh_<FAST>(d2 * za + bb);
      za += d1 * th;
    }
    // ---- rgb stack (z_size 3; components reversed on odd flows, models.py:404-408): flow_composite.cu:149-164 ----
    float z0c = z0.x, z1c = z0.y, z2c = z0.z;
#pragma unroll
    for (int f = 0; f < F; ++f) {
      const float* Q = P + 3 * F + kRgbFlowRec * f;
      const bool odd = f & 1;
      const float q0 = odd ? z2c : z0c, q1 = z1c, q2 = odd ? z0c : z2c;
      const float t0 = tanh_<FAST>(Q[6] * q0 + Q[7] * q1 + Q[8] * q2 + Q[12]);
      const float t1 = tanh_<FAST>(Q[9] * q1 + Q[10] * q2 + Q[13]);
      const float t2 = tanh_<FAST>(Q[11] * q2 + Q[14]);
      const float s0 = Q[0] * t0 + Q[1] * t1 + Q[2] * t2;
      const float s1 = Q[3] * t1 + Q[4] * t2;
      const float s2 = Q[5] * t2;
      z0c += odd ? s2 : s0;
      z1c += s1;
      z2c += odd ? s0 : s2;
    }
    const float inv = sinv[k];
    welford(softplus_<FAST>(za), inv, s_mean, s_m2);
    welford(sigmoid_<FAST>(z0c), inv, r_mean, r_m2);
    welford(sigmoid_<FAST>(z1c), inv, g_mean, g_m2);
    welford(sigmoid_<FAST>(z2c), inv, b_mean, b_m2);
  }
  const float inv_km1 = K > 1 ? 1.0f / (float)(K - 1) : 0.f;
  float4* o = reinterpret_cast<float4*>(out + (p0 + t) * 8);
  o[0] = make_float4(s_mean, sqrtf(s_m2 * inv_km1), r_mean, g_mean);
  o[1] = make_float4(b_mean, sqrtf(r_m2 * inv_km1), sqrtf(g_m2 * inv_km1), sqrtf(b_m2 * inv_km1));
}

static size_t field_smem_bytes(int F, int K) { return ((size_t)5 * K + (size_t)kFieldThreads * (18 * F + 1)) * sizeof(float); }

int launch_field_stats(int fast_math, int F, int K, const float* globals, const float* flow_params, const float* eps_alpha,
                       const float* eps_rgb, int64_t M, float* out, cudaStream_t s) {
  if (M == 0) return CFN_OK;
  CFN_CHECK_ARG(F >= 1 && F <= 8 && K >= 1 && K <= 1024, "field_stats: unsupported F=%d K=%d (1..8, 1..1024)", F, K);
  const size_t smem = field_smem_bytes(F, K);
  const unsigned grid = (unsigned)((M + kFieldThreads - 1) / kFieldThreads);
#define CFN_FIELD_LAUNCH(FASTM, FTT)                                                                                  \
  do {                                                                                                               \
    auto kern = field_stats_kernel<FASTM, FTT>;                                                                      \
    if (smem > 48 * 1024) CFN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kern<<<grid, kFieldThreads, smem, s>>>(F, K, globals, flow_params, eps_alpha, eps_rgb, M, out);                  \
  } while (0)
  if (fast_math) { if (F == 4) CFN_FIELD_LAUNCH(true, 4); else CFN_FIELD_LAUNCH(true, 0); }
  else { if (F == 4) CFN_FIELD_LAUNCH(false, 4); else CFN_FIELD_LAUNCH(false, 0); }
#undef CFN_FIELD_LAUNCH
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

}  // namespace cfn
