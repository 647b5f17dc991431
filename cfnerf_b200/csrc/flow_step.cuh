// The per-point flow step and the per-sample compositing update of one latent draw for the flow warps of the fused
// network kernel (mlp_tc.cu): the operations of K2's render flavour (flow_composite_fwd_kernel) in the same order, so the
// maps the fused kernel writes are bitwise equal to K1 -> K2 (tests/test_fused_composite.py).  K2 keeps its own inline
// copy: compiled through these functions it ran 6.5 % slower on a B200 (0.817 -> 0.870 ms per 16 384 rays at K = 32).
//
// Reference semantics: model/models.py:188-291 + 387-416 (flow stacks), run_nerf_uncertainty_NF.py:411-454
// (raw2outputs).
#pragma once
#include "common.cuh"

namespace cfn {

// alpha stack (z_size 1; the flip is the identity).  P: the point's record.
template <bool FAST>
__device__ __forceinline__ float flow_alpha(const float* P, int F, float za) {
#pragma unroll
  for (int f = 0; f < F; ++f) {
    const float d1 = P[f], d2 = P[F + f], bb = P[2 * F + f];
    const float t = tanh_<FAST>(d2 * za + bb);
    za += d1 * t;
  }
  return za;
}

// rgb stack (z_size 3; components reversed on odd flows, models.py:404-408), in place on (z0, z1, z2)
template <bool FAST>
__device__ __forceinline__ void flow_rgb(const float* P, int F, float& z0, float& z1, float& z2) {
#pragma unroll
  for (int f = 0; f < F; ++f) {
    const float* Q = P + 3 * F + kRgbFlowRec * f;
    const bool odd = f & 1;
    const float p0 = odd ? z2 : z0, p1 = z1, p2 = odd ? z0 : z2;
    const float t0 = tanh_<FAST>(Q[6] * p0 + Q[7] * p1 + Q[8] * p2 + Q[12]);
    const float t1 = tanh_<FAST>(Q[9] * p1 + Q[10] * p2 + Q[13]);
    const float t2 = tanh_<FAST>(Q[11] * p2 + Q[14]);
    const float s0 = Q[0] * t0 + Q[1] * t1 + Q[2] * t2;
    const float s1 = Q[3] * t1 + Q[4] * t2;
    const float s2 = Q[5] * t2;
    z0 += odd ? s2 : s0;
    z1 += s1;
    z2 += odd ? s0 : s2;
  }
}

// Front-to-back state of one (ray, latent draw) and the compositing of one sample at depth z, `dist` = delta * |d|
struct RayAcc {
  float T = 1.0f, cr = 0.f, cg = 0.f, cb = 0.f, depth = 0.f, acc = 0.f;
};
template <bool FAST>
__device__ __forceinline__ void composite_sample(RayAcc& r, float za, float z0, float z1, float z2, float z, float dist) {
  const float alpha = 1.0f - exp_<FAST>(-softplus_<FAST>(za) * dist);
  const float w = alpha * r.T;
  r.T = r.T * ((1.0f - alpha) + 1e-10f);
  const float wc0 = w * sigmoid_<FAST>(z0), wc1 = w * sigmoid_<FAST>(z1), wc2 = w * sigmoid_<FAST>(z2), wz = w * z;
  r.cr += wc0;
  r.cg += wc1;
  r.cb += wc2;
  r.depth += wz;
  r.acc += w;
}

// disparity and white background of a finished ray; the maps of draw k (active lanes) and the kstats sums
__device__ __forceinline__ void finish_ray(RayAcc& r, int white_bkgd, bool active, int64_t b, int K, int k, float* rgb_map,
                                           float* disp_map, float* depth_map, float (&st_sum)[5]) {
  const float disp = 1.0f / fmaxf(2e-10f, r.depth / (r.acc + 1e-10f) + 1e-10f);
  if (white_bkgd) {
    const float bg = 1.0f - r.acc;
    r.cr += bg; r.cg += bg; r.cb += bg;
  }
  if (active) {
    rgb_map[(b * 3 + 0) * K + k] = r.cr;
    rgb_map[(b * 3 + 1) * K + k] = r.cg;
    rgb_map[(b * 3 + 2) * K + k] = r.cb;
    disp_map[b * K + k] = disp;
    depth_map[b * K + k] = r.depth;
    st_sum[0] += r.cr; st_sum[1] += r.cg; st_sum[2] += r.cb; st_sum[3] += r.depth; st_sum[4] += disp;
  }
}

// kstats of ray b (whole warp, after every K group): mean over K, then the centred second moment from the colours this
// warp just wrote (L1 / L2 hits)
__device__ __forceinline__ void write_kstats(int64_t b, int K, int lane, const float* rgb_map, float (&st_sum)[5],
                                             float* kstats) {
  float st_sq[3] = {0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 5; ++j)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) st_sum[j] += __shfl_xor_sync(0xffffffffu, st_sum[j], o);
  const float invK = 1.0f / (float)K;
  const float m0 = st_sum[0] * invK, m1 = st_sum[1] * invK, m2 = st_sum[2] * invK;
  __syncwarp();
  for (int k = lane; k < K; k += 32) {
    const float a0 = rgb_map[(b * 3 + 0) * K + k] - m0, a1 = rgb_map[(b * 3 + 1) * K + k] - m1,
                a2 = rgb_map[(b * 3 + 2) * K + k] - m2;
    st_sq[0] += a0 * a0; st_sq[1] += a1 * a1; st_sq[2] += a2 * a2;
  }
#pragma unroll
  for (int j = 0; j < 3; ++j)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) st_sq[j] += __shfl_xor_sync(0xffffffffu, st_sq[j], o);
  if (lane == 0) {
    const float bess = (K > 1) ? (float)K / (float)(K - 1) : 0.f;       // the second K/(K-1) factor (main:1034)
    const float inv = (K > 1) ? 1.0f / (float)(K - 1) : 0.f;
    float* o = kstats + b * 8;
    o[0] = m0; o[1] = m1; o[2] = m2;
    o[3] = sqrtf(st_sq[0] * inv) * bess;
    o[4] = sqrtf(st_sq[1] * inv) * bess;
    o[5] = sqrtf(st_sq[2] * inv) * bess;
    o[6] = st_sum[3] * invK;
    o[7] = st_sum[4] * invK;
  }
}

}  // namespace cfn
