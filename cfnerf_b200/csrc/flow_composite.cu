// K2 / K4: conditional triangular-Sylvester flow stacks over K latent samples + alpha compositing of all K
// fields, forward and backward.  One warp per ray, lane = latent sample k (groups of 32 when K > 32); the warp
// walks the N samples front to back, carrying transmittance and the running sums in registers, so there is no
// scan primitive and no (B,N,K,...) intermediate in HBM.  The 18F conditioning scalars of each point are staged
// through shared memory in 16-point chunks (coalesced 128-bit loads, register double-buffering) and read back
// as warp-wide broadcasts.
//
// Reference semantics: model/models.py:188-291 (NeRF_Flows.forward), model/models.py:387-416 +
// model/flow/flows.py:189-268 (flow step, log-det), run_nerf_uncertainty_NF.py:411-454 (raw2outputs);
// backward = SURVEY.md Appendix A.1/A.2 (verified there against autograd).
#include "common.cuh"

namespace cfn {

constexpr int kChunk = 16;   // points staged per shared-memory chunk
constexpr int kMaxF = 8;     // flows per stack supported by the backward kernel's register arrays

// Stage one chunk of flow parameters: global (coalesced) -> registers.
template <int MAXV>
__device__ __forceinline__ void chunk_load(const float* __restrict__ src, int n_floats, int lane, float4 (&v)[MAXV]) {
  const int nvec = n_floats >> 2;  // chunk base is 16-byte aligned (16*PP floats per chunk)
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int idx = lane + 32 * i;
    if (idx < nvec) v[i] = __ldg(reinterpret_cast<const float4*>(src) + idx);
  }
}
template <int MAXV>
__device__ __forceinline__ void chunk_store(float* dst, int n_floats, int lane, const float4 (&v)[MAXV]) {
  const int nvec = n_floats >> 2;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int idx = lane + 32 * i;
    if (idx < nvec) reinterpret_cast<float4*>(dst)[idx] = v[i];
  }
}

// MAXV float4 per lane must cover kChunk*PP/4 float4 per chunk: PP = 18F -> 72F float4 / 32 lanes.
// F <= 8 -> at most 18 float4 per lane.  We instantiate for F<=4 (MAXV=9) and F<=8 (MAXV=18).

template <int MAXV, bool TRAIN, bool FAST, int FT>
__global__ void __launch_bounds__(128, 4)   // 16 warps per SM: the kernel is latency / issue bound, occupancy is what it needs
flow_composite_fwd_kernel(int F_rt, int K, const float* __restrict__ globals, const float* __restrict__ flow_params,
                          const float* __restrict__ z_vals, const float* __restrict__ rays_d, int rays_d_stride,
                          const float* __restrict__ eps_alpha, const float* __restrict__ eps_rgb,
                          int64_t eps_group_rays, int64_t B, int N,
                          int white_bkgd, float* __restrict__ rgb_map, float* __restrict__ disp_map,
                          float* __restrict__ depth_map, float* __restrict__ raw, float* __restrict__ weights,
                          float* __restrict__ logdet_sums, float* __restrict__ kstats, float* __restrict__ trans,
                          float* __restrict__ seg_sums, int n_seg) {
  extern __shared__ __align__(16) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // FT > 0: the number of flows is a compile-time constant (the shipped recipe, F = 4): a point's 18F scalars are
  // read as 128-bit shared-memory broadcasts into registers and every flow loop is unrolled
  const int F = FT > 0 ? FT : F_rt;
  const int PP = 18 * F;
  const int per_warp = (kChunk * PP + 2 * N + 3) & ~3;   // keeps every warp's chunk buffer 16-byte aligned
  float* sp = smem + warp * per_warp;  // chunk of parameters
  float* sz = sp + kChunk * PP;        // z_vals of the ray
  float* sd = sz + N;                  // dists * |d|
  const int64_t b = (int64_t)blockIdx.x * 4 + warp;
  if (b >= B) return;
  // base latent draws: one (K) / (K,3) set per group of eps_group_rays consecutive rays (the reference draws fresh noise
  // in every network call of netchunk points, models.py:233-251; 0 = one set shared by all rays)
  const int64_t egrp = eps_group_rays > 0 ? b / eps_group_rays : 0;
  eps_alpha += egrp * K;
  eps_rgb += egrp * K * 3;

  for (int n = lane; n < N; n += 32) sz[n] = z_vals[b * N + n];
  const float* d = rays_d + b * rays_d_stride;
  const float dx = d[0], dy = d[1], dz = d[2];
  const float norm = sqrtf(dx * dx + dy * dy + dz * dz);
  __syncwarp();
  for (int n = lane; n < N; n += 32) sd[n] = ((n < N - 1) ? (sz[n + 1] - sz[n]) : 10.0f) * norm;

  const float a_mean = globals[0], a_std = globals[1];
  const float c_mean0 = globals[2], c_mean1 = globals[3], c_mean2 = globals[4];
  const float c_std0 = globals[5], c_std1 = globals[6], c_std2 = globals[7];

  const float* prow = flow_params + (b * N) * PP;
  const int n_chunks = (N + kChunk - 1) / kChunk;
  const int KG = (K + 31) / 32;
  // 128-bit staging needs a 16-byte aligned row (always true for even N*F); otherwise everything goes scalar
  const bool vec_ok = (reinterpret_cast<uintptr_t>(prow) & 15) == 0;

  float ld_a_sum = 0.f, ld_c_sum = 0.f;                      // TRAIN: per-lane sums of the log-det terms
  float st_sum[5] = {0.f, 0.f, 0.f, 0.f, 0.f};               // kstats: sums over k of r,g,b,depth,disp
  float st_sq[3] = {0.f, 0.f, 0.f};

  // two passes over the K groups when kstats needs a centred variance: we keep it single pass and use the
  // shifted two-accumulator form below only for K <= 32 groups; variance is finalised after the loop.
  for (int kg = 0; kg < KG; ++kg) {
    const int k = kg * 32 + lane;
    const bool active = k < K;
    const float ea = active ? eps_alpha[k] : 0.f;
    const float e0 = active ? eps_rgb[k * 3 + 0] : 0.f, e1 = active ? eps_rgb[k * 3 + 1] : 0.f,
                e2 = active ? eps_rgb[k * 3 + 2] : 0.f;
    // z0 = eps * std + mean  (models.py:200/206, 239/251)
    const float za0 = ea * a_std + a_mean;
    const float zc00 = e0 * c_std0 + c_mean0, zc01 = e1 * c_std1 + c_mean1, zc02 = e2 * c_std2 + c_mean2;

    float T = 1.0f, cr = 0.f, cg = 0.f, cb = 0.f, depth = 0.f, acc = 0.f;
    // TRAIN, n_seg > 1: sums of w*c (3), w*z, w over each of the n_seg equal sample ranges of the ray, written as
    // seg_sums[b][seg][5][K].  The backward splits a ray into n_seg independent warps: the one that owns range s starts
    // its suffix-sum recurrence from the (cancellation-free: all terms are non-negative) sums of the later ranges.
    float sg0 = 0.f, sg1 = 0.f, sg2 = 0.f, sg3 = 0.f, sg4 = 0.f;
    const int seg_len = (TRAIN && seg_sums && n_seg > 1) ? N / n_seg : 0;
    int seg_left = seg_len, seg_idx = 0;

    float4 stage[MAXV];
    {
      const int npts = min(kChunk, N);
      const int nvf = vec_ok ? ((npts * PP) & ~3) : 0;
      chunk_load<MAXV>(prow, nvf, lane, stage);
      __syncwarp();
      chunk_store<MAXV>(sp, nvf, lane, stage);
      for (int i = nvf + lane; i < npts * PP; i += 32) sp[i] = prow[i];   // scalar tail / unaligned rows
      __syncwarp();
    }
    for (int c = 0; c < n_chunks; ++c) {
      const int n0 = c * kChunk;
      const int npts = min(kChunk, N - n0);
      const bool has_next = (c + 1) < n_chunks;
      const int next_pts = has_next ? min(kChunk, N - n0 - kChunk) : 0;
      const int next_vf = vec_ok ? ((next_pts * PP) & ~3) : 0;
      if (has_next) chunk_load<MAXV>(prow + (int64_t)(n0 + kChunk) * PP, next_vf, lane, stage);

      for (int i = 0; i < npts; ++i) {
        const int n = n0 + i;
        float rec[FT > 0 ? 18 * FT : 4];
        const float* P = sp + i * PP;
        if (FT > 0) {
#pragma unroll
          for (int j = 0; j < (18 * FT) / 4; ++j) {
            const float4 q4 = reinterpret_cast<const float4*>(sp + i * PP)[j];
            rec[4 * j] = q4.x; rec[4 * j + 1] = q4.y; rec[4 * j + 2] = q4.z; rec[4 * j + 3] = q4.w;
          }
          P = rec;
        }
        // ---- alpha stack (z_size 1; the flip is the identity) ----
        float za = za0, lda = 0.f;
#pragma unroll
        for (int f = 0; f < F; ++f) {
          const float d1 = P[f], d2 = P[F + f], bb = P[2 * F + f];
          const float t = tanh_<FAST>(d2 * za + bb);
          za += d1 * t;
          if (TRAIN) lda += log_<FAST>(fabsf((1.0f - t * t) * (d1 * d2) + 1.0f) + 1e-8f);
        }
        // ---- rgb stack (z_size 3; components reversed on odd flows, models.py:404-408) ----
        float z0 = zc00, z1 = zc01, z2 = zc02, ldc = 0.f;
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
          if (TRAIN) {
            ldc += log_<FAST>(fabsf((1.0f - t0 * t0) * (Q[0] * Q[6]) + 1.0f) + 1e-8f) +
                   log_<FAST>(fabsf((1.0f - t1 * t1) * (Q[3] * Q[9]) + 1.0f) + 1e-8f) +
                   log_<FAST>(fabsf((1.0f - t2 * t2) * (Q[5] * Q[11]) + 1.0f) + 1e-8f);
          }
        }
        if (TRAIN && active) {
          ld_a_sum += lda + (za - softplus_<FAST>(za));                                           // models.py:263
          ld_c_sum += ldc + ((z0 + z1 + z2) - 2.0f * (softplus_<FAST>(z0) + softplus_<FAST>(z1) + softplus_<FAST>(z2)));  // :278
        }
        // ---- compositing (raw2outputs) ----
        const float alpha = 1.0f - exp_<FAST>(-softplus_<FAST>(za) * sd[n]);
        const float w = alpha * T;
        if (TRAIN && trans && active) trans[(b * N + n) * K + k] = T;   // transmittance in front of sample n (K4 reads it)
        T = T * ((1.0f - alpha) + 1e-10f);
        const float wc0 = w * sigmoid_<FAST>(z0), wc1 = w * sigmoid_<FAST>(z1), wc2 = w * sigmoid_<FAST>(z2), wz = w * sz[n];
        cr += wc0;
        cg += wc1;
        cb += wc2;
        depth += wz;
        acc += w;
        if (TRAIN && seg_len) {
          sg0 += wc0; sg1 += wc1; sg2 += wc2; sg3 += wz; sg4 += w;
          if (--seg_left == 0) {
            if (active) {
              float* o = seg_sums + ((b * n_seg + seg_idx) * 5) * K + k;
              o[0] = sg0; o[K] = sg1; o[2 * K] = sg2; o[3 * K] = sg3; o[4 * K] = sg4;
            }
            sg0 = sg1 = sg2 = sg3 = sg4 = 0.f;
            seg_left = seg_len; ++seg_idx;
          }
        }
        if (active) {
          if (raw) reinterpret_cast<float4*>(raw)[(b * N + n) * K + k] = make_float4(z0, z1, z2, za);
          if (weights) weights[(b * N + n) * K + k] = w;
        }
      }
      __syncwarp();
      if (has_next) {
        chunk_store<MAXV>(sp, next_vf, lane, stage);
        const float* src = prow + (int64_t)(n0 + kChunk) * PP;
        for (int i = next_vf + lane; i < next_pts * PP; i += 32) sp[i] = src[i];
      }
      __syncwarp();
    }
    const float disp = 1.0f / fmaxf(2e-10f, depth / (acc + 1e-10f) + 1e-10f);
    if (white_bkgd) {
      const float bg = 1.0f - acc;
      cr += bg; cg += bg; cb += bg;
    }
    if (active) {
      rgb_map[(b * 3 + 0) * K + k] = cr;
      rgb_map[(b * 3 + 1) * K + k] = cg;
      rgb_map[(b * 3 + 2) * K + k] = cb;
      disp_map[b * K + k] = disp;
      depth_map[b * K + k] = depth;
      st_sum[0] += cr; st_sum[1] += cg; st_sum[2] += cb; st_sum[3] += depth; st_sum[4] += disp;
    }
  }

  if (TRAIN && logdet_sums) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      ld_a_sum += __shfl_xor_sync(0xffffffffu, ld_a_sum, o);
      ld_c_sum += __shfl_xor_sync(0xffffffffu, ld_c_sum, o);
    }
    if (lane == 0) {
      logdet_sums[b * 2 + 0] = ld_a_sum;
      logdet_sums[b * 2 + 1] = ld_c_sum;
    }
  }
  if (kstats) {
    // mean over K, then the centred second moment from the values just written (L1/L2 hits)
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
}

// ---------------------------------------------------------------------------------------------------------------
// Training forward for SMALL batches: one CTA of 4 warps per ray, warp s walks samples [s N/4, (s+1) N/4).
// With one warp per ray a 512-ray batch (the reference's N_rand) occupies 512 of the 2 368 warp slots of a B200 and each
// warp walks 128 dependent samples: the kernel is pure latency (0.114 ms for 512 rays against 0.37 ms for 4096).  The
// flow stacks - all of the cost - are independent per sample; only the transmittance chains them.  Every warp therefore
// starts its range at T = 1; the true transmittance is (product of the earlier ranges' final T) x local T, applied
// afterwards to the range sums (exactly the seg_sums the backward wants), to the outputs and, in place, to `trans`.
// Same arithmetic per sample as flow_composite_fwd_kernel<TRAIN = true>; the transmittance products associate
// differently (relative difference ~1e-7).
template <int MAXV, bool FAST, int FT>
__global__ void __launch_bounds__(128, 4)
flow_composite_fwd_seg4_kernel(int F_rt, int K, const float* __restrict__ globals, const float* __restrict__ flow_params,
                               const float* __restrict__ z_vals, const float* __restrict__ rays_d, int rays_d_stride,
                               const float* __restrict__ eps_alpha, const float* __restrict__ eps_rgb,
                               int64_t eps_group_rays, int64_t B, int N, int white_bkgd, float* __restrict__ rgb_map,
                               float* __restrict__ disp_map, float* __restrict__ depth_map, float* __restrict__ raw,
                               float* __restrict__ logdet_sums, float* __restrict__ trans, float* __restrict__ seg_sums) {
  extern __shared__ __align__(16) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int F = FT > 0 ? FT : F_rt;
  const int PP = 18 * F;
  const int per_warp = (kChunk * PP + 3) & ~3;
  float* sp = smem + warp * per_warp;                 // this warp's chunk of parameters
  float* sz = smem + 4 * per_warp;                    // z_vals of the ray (shared by the four warps)
  float* sd = sz + N;                                 // dists * |d|
  float* sP = sd + N;                                 // [4][32] final local transmittance of each range
  float* sS = sP + 4 * 32;                            // [4][5][32] scaled range sums
  float* sL = sS + 4 * 5 * 32;                        // [4][2] log-det sums
  const int64_t b = blockIdx.x;
  const int64_t egrp = eps_group_rays > 0 ? b / eps_group_rays : 0;
  eps_alpha += egrp * K;
  eps_rgb += egrp * K * 3;
  for (int n = threadIdx.x; n < N; n += 128) sz[n] = z_vals[b * N + n];
  const float* d = rays_d + b * rays_d_stride;
  const float dx = d[0], dy = d[1], dz = d[2];
  const float norm = sqrtf(dx * dx + dy * dy + dz * dz);
  __syncthreads();
  for (int n = threadIdx.x; n < N; n += 128) sd[n] = ((n < N - 1) ? (sz[n + 1] - sz[n]) : 10.0f) * norm;
  __syncthreads();

  const float a_mean = globals[0], a_std = globals[1];
  const float c_mean0 = globals[2], c_mean1 = globals[3], c_mean2 = globals[4];
  const float c_std0 = globals[5], c_std1 = globals[6], c_std2 = globals[7];
  const int L = N / 4, n_begin = warp * L;
  const float* prow = flow_params + (b * N + n_begin) * PP;
  const int n_chunks = (L + kChunk - 1) / kChunk;
  const int KG = (K + 31) / 32;
  const bool vec_ok = (reinterpret_cast<uintptr_t>(prow) & 15) == 0;
  float ld_a_sum = 0.f, ld_c_sum = 0.f;

  for (int kg = 0; kg < KG; ++kg) {
    const int k = kg * 32 + lane;
    const bool active = k < K;
    const float ea = active ? eps_alpha[k] : 0.f;
    const float e0 = active ? eps_rgb[k * 3 + 0] : 0.f, e1 = active ? eps_rgb[k * 3 + 1] : 0.f,
                e2 = active ? eps_rgb[k * 3 + 2] : 0.f;
    const float za0 = ea * a_std + a_mean;
    const float zc00 = e0 * c_std0 + c_mean0, zc01 = e1 * c_std1 + c_mean1, zc02 = e2 * c_std2 + c_mean2;
    float T = 1.0f, cr = 0.f, cg = 0.f, cb = 0.f, depth = 0.f, acc = 0.f;

    float4 stage[MAXV];
    {
      const int npts = min(kChunk, L);
      const int nvf = vec_ok ? ((npts * PP) & ~3) : 0;
      chunk_load<MAXV>(prow, nvf, lane, stage);
      __syncwarp();
      chunk_store<MAXV>(sp, nvf, lane, stage);
      for (int i = nvf + lane; i < npts * PP; i += 32) sp[i] = prow[i];
      __syncwarp();
    }
    for (int c = 0; c < n_chunks; ++c) {
      const int n0 = c * kChunk;
      const int npts = min(kChunk, L - n0);
      const bool has_next = (c + 1) < n_chunks;
      const int next_pts = has_next ? min(kChunk, L - n0 - kChunk) : 0;
      const int next_vf = vec_ok ? ((next_pts * PP) & ~3) : 0;
      if (has_next) chunk_load<MAXV>(prow + (int64_t)(n0 + kChunk) * PP, next_vf, lane, stage);
      for (int i = 0; i < npts; ++i) {
        const int n = n_begin + n0 + i;
        float rec[FT > 0 ? 18 * FT : 4];
        const float* P = sp + i * PP;
        if (FT > 0) {
#pragma unroll
          for (int j = 0; j < (18 * FT) / 4; ++j) {
            const float4 q4 = reinterpret_cast<const float4*>(sp + i * PP)[j];
            rec[4 * j] = q4.x; rec[4 * j + 1] = q4.y; rec[4 * j + 2] = q4.z; rec[4 * j + 3] = q4.w;
          }
          P = rec;
        }
        float za = za0, lda = 0.f;
#pragma unroll
        for (int f = 0; f < F; ++f) {
          const float d1 = P[f], d2 = P[F + f], bb = P[2 * F + f];
          const float t = tanh_<FAST>(d2 * za + bb);
          za += d1 * t;
          lda += log_<FAST>(fabsf((1.0f - t * t) * (d1 * d2) + 1.0f) + 1e-8f);
        }
        float z0 = zc00, z1 = zc01, z2 = zc02, ldc = 0.f;
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
          ldc += log_<FAST>(fabsf((1.0f - t0 * t0) * (Q[0] * Q[6]) + 1.0f) + 1e-8f) +
                 log_<FAST>(fabsf((1.0f - t1 * t1) * (Q[3] * Q[9]) + 1.0f) + 1e-8f) +
                 log_<FAST>(fabsf((1.0f - t2 * t2) * (Q[5] * Q[11]) + 1.0f) + 1e-8f);
        }
        if (active) {
          ld_a_sum += lda + (za - softplus_<FAST>(za));                                           // models.py:263
          ld_c_sum += ldc + ((z0 + z1 + z2) - 2.0f * (softplus_<FAST>(z0) + softplus_<FAST>(z1) + softplus_<FAST>(z2)));  // :278
        }
        const float alpha = 1.0f - exp_<FAST>(-softplus_<FAST>(za) * sd[n]);
        const float w = alpha * T;
        if (active) trans[(b * N + n) * K + k] = T;          // LOCAL transmittance for now; rescaled below
        T = T * ((1.0f - alpha) + 1e-10f);
        cr += w * sigmoid_<FAST>(z0);
        cg += w * sigmoid_<FAST>(z1);
        cb += w * sigmoid_<FAST>(z2);
        depth += w * sz[n];
        acc += w;
        if (active && raw) reinterpret_cast<float4*>(raw)[(b * N + n) * K + k] = make_float4(z0, z1, z2, za);
      }
      __syncwarp();
      if (has_next) {
        chunk_store<MAXV>(sp, next_vf, lane, stage);
        const float* src = prow + (int64_t)(n0 + kChunk) * PP;
        for (int i = next_vf + lane; i < next_pts * PP; i += 32) sp[i] = src[i];
      }
      __syncwarp();
    }
    // ---- stitch the four ranges together ----
    sP[warp * 32 + lane] = T;
    __syncthreads();
    float prefix = 1.0f;
    for (int s2 = 0; s2 < warp; ++s2) prefix *= sP[s2 * 32 + lane];
    cr *= prefix; cg *= prefix; cb *= prefix; depth *= prefix; acc *= prefix;
    if (active) {
      float* o = seg_sums + ((b * 4 + warp) * 5) * K + k;
      o[0] = cr; o[K] = cg; o[2 * K] = cb; o[3 * K] = depth; o[4 * K] = acc;
      if (warp > 0)
        for (int n = n_begin; n < n_begin + L; ++n) trans[(b * N + n) * K + k] *= prefix;   // own writes: L1 / L2 hits
    }
    float* my = sS + warp * 160;
    my[lane] = cr; my[32 + lane] = cg; my[64 + lane] = cb; my[96 + lane] = depth; my[128 + lane] = acc;
    __syncthreads();
    if (warp == 0 && active) {
      float tr = 0.f, tg = 0.f, tb = 0.f, td = 0.f, ta = 0.f;
#pragma unroll
      for (int s2 = 0; s2 < 4; ++s2) {
        const float* q = sS + s2 * 160;
        tr += q[lane]; tg += q[32 + lane]; tb += q[64 + lane]; td += q[96 + lane]; ta += q[128 + lane];
      }
      const float disp = 1.0f / fmaxf(2e-10f, td / (ta + 1e-10f) + 1e-10f);
      if (white_bkgd) { const float bg = 1.0f - ta; tr += bg; tg += bg; tb += bg; }
      rgb_map[(b * 3 + 0) * K + k] = tr;
      rgb_map[(b * 3 + 1) * K + k] = tg;
      rgb_map[(b * 3 + 2) * K + k] = tb;
      disp_map[b * K + k] = disp;
      depth_map[b * K + k] = td;
    }
    __syncthreads();     // sP / sS are reused by the next K group
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ld_a_sum += __shfl_xor_sync(0xffffffffu, ld_a_sum, o);
    ld_c_sum += __shfl_xor_sync(0xffffffffu, ld_c_sum, o);
  }
  if (lane == 0) { sL[warp * 2] = ld_a_sum; sL[warp * 2 + 1] = ld_c_sum; }
  __syncthreads();
  if (threadIdx.x == 0) {
    logdet_sums[b * 2 + 0] = (sL[0] + sL[2]) + (sL[4] + sL[6]);
    logdet_sums[b * 2 + 1] = (sL[1] + sL[3]) + (sL[5] + sL[7]);
  }
}

static size_t fwd_smem_bytes(int F, int N) { return (size_t)4 * ((kChunk * 18 * F + 2 * N + 3) & ~3) * sizeof(float); }

int launch_flow_composite_fwd(int fast_math, int F, int K, const float* globals, const float* flow_params, const float* z_vals,
                              const float* rays_d, int rays_d_stride, const float* eps_alpha, const float* eps_rgb,
                              int64_t eps_group_rays, int64_t B, int N, int white_bkgd, float* rgb_map, float* disp_map,
                              float* depth_map, float* raw, float* weights, float* logdet_sums, float* kstats, float* trans,
                              float* seg_sums, int n_seg, cudaStream_t s) {
  if (B == 0) return CFN_OK;
  CFN_CHECK_ARG(!seg_sums || (n_seg >= 1 && N % n_seg == 0), "flow_composite: N=%d is not a multiple of n_segments=%d", N, n_seg);
  CFN_CHECK_ARG(F >= 1 && F <= kMaxF, "flow_composite: n_flows=%d unsupported (1..%d)", F, kMaxF);
  CFN_CHECK_ARG(N >= 1 && N <= 2048 && K >= 1, "flow_composite: unsupported N=%d K=%d (need 1 <= N <= 2048)", N, K);
  size_t smem = fwd_smem_bytes(F, N);
  unsigned grid = (unsigned)((B + 3) / 4);
  const bool train = logdet_sums != nullptr;
  // small training batches: four warps per ray (see flow_composite_fwd_seg4_kernel)
  if (train && trans && seg_sums && n_seg == 4 && N % 4 == 0 && !weights && !kstats && B <= 1536 && F <= 4) {
    const size_t sm4 = ((size_t)4 * ((kChunk * 18 * F + 3) & ~3) + 2 * (size_t)N + 4 * 32 + 4 * 5 * 32 + 8) * sizeof(float);
#define CFN_SEG4_LAUNCH(FASTM, FTT)                                                                                  \
    do {                                                                                                             \
      auto kern = flow_composite_fwd_seg4_kernel<9, FASTM, FTT>;                                                     \
      if (sm4 > 48 * 1024) CFN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm4)); \
      kern<<<(unsigned)B, 128, sm4, s>>>(F, K, globals, flow_params, z_vals, rays_d, rays_d_stride, eps_alpha, eps_rgb, \
                                         eps_group_rays, B, N, white_bkgd, rgb_map, disp_map, depth_map, raw,        \
                                         logdet_sums, trans, seg_sums);                                              \
    } while (0)
    if (fast_math) { if (F == 4) CFN_SEG4_LAUNCH(true, 4); else CFN_SEG4_LAUNCH(true, 0); }
    else { if (F == 4) CFN_SEG4_LAUNCH(false, 4); else CFN_SEG4_LAUNCH(false, 0); }
#undef CFN_SEG4_LAUNCH
    CFN_LAUNCH_CHECK();
    return CFN_OK;
  }
#define CFN_FWD_LAUNCH(MAXV, TR)                                                                                  \
  do {                                                                                                            \
    auto kern = fast_math ? (F == 4 ? flow_composite_fwd_kernel<MAXV, TR, true, 4> : flow_composite_fwd_kernel<MAXV, TR, true, 0>)\
                          : (F == 4 ? flow_composite_fwd_kernel<MAXV, TR, false, 4> : flow_composite_fwd_kernel<MAXV, TR, false, 0>);                                                            \
    if (smem > 48 * 1024) CFN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kern<<<grid, 128, smem, s>>>(F, K, globals, flow_params, z_vals, rays_d, rays_d_stride, eps_alpha, eps_rgb,   \
                                 eps_group_rays, B, N, white_bkgd, rgb_map, disp_map, depth_map, raw, weights,    \
                                 logdet_sums, kstats, trans, seg_sums, n_seg);                                    \
  } while (0)
  if (F <= 4) {
    if (train) CFN_FWD_LAUNCH(9, true); else CFN_FWD_LAUNCH(9, false);
  } else {
    if (train) CFN_FWD_LAUNCH(18, true); else CFN_FWD_LAUNCH(18, false);
  }
#undef CFN_FWD_LAUNCH
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

// =====================================================================================================
// Backward (K4).  One warp per ray, lane = latent sample k, ONE pass back to front:
//   * the transmittance T_n in front of every sample comes from HBM (B,N,K): the training forward writes it for free
//     (K2 `trans` output).  Keeping it in shared memory (round 1: N x 32 floats per warp) capped the kernel at 8 warps per SM, and at ~1200 dependent
//     instructions per point the kernel is latency bound: occupancy is what it needs;
//   * per point both stacks are recomputed with their intermediates in registers, the compositing adjoint carries the
//     suffix sum S (Appendix A.2), the flow adjoints run step by step in reverse (Appendix A.1);
//   * the 18F per-point parameter gradients are reduced over the 32 latent lanes 16 rows at a time through a small
//     double-buffered shared-memory scratch (16 x 36 floats: conflict-free column stores, two lanes per row read four
//     float4 each, one shuffle joins the halves) — one __syncwarp per 16 rows, 4.5 KB per warp instead of 10 KB;
//   * parameters are staged PB points at a time (coalesced loads, register prefetch of the next block) and the reduced
//     gradient rows of a block leave through shared memory as contiguous stores.
// Gradients w.r.t. the global latent parameters through z0 = eps*std + mean are summed per ray into
// g_globals_partial (B,8) (deterministic; the host sums over rays).
// =====================================================================================================
constexpr int kBwdPB = 4;     // points per staged block
constexpr int kBwdGLD = 36;   // row stride of the reduction scratch: 32 lanes + 4 (rows stay 16-byte aligned, no conflicts)

// sum v[0..NV) over the 32 lanes, 16 rows per round; row r of round g0 lands in out[g0 + r]
template <int NV>
__device__ __forceinline__ void reduce_rows_over_lanes(const float (&v)[NV], float* __restrict__ sG, int& buf,
                                                       float* __restrict__ out, int lane) {
  const int row = lane >> 1, half = lane & 1;
#pragma unroll
  for (int g0 = 0; g0 < NV; g0 += 16) {
    constexpr int kRows = 16;
    const int cnt = (NV - g0 < kRows) ? (NV - g0) : kRows;
    float* S = sG + buf * (16 * kBwdGLD);
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (g0 + i < NV) S[i * kBwdGLD + lane] = v[g0 + i];
    __syncwarp();
    float acc = 0.f;
    if (row < cnt) {
      const float4* r4 = reinterpret_cast<const float4*>(S + row * kBwdGLD + half * 16);
      const float4 a = r4[0], b4 = r4[1], c = r4[2], d = r4[3];
      acc = ((a.x + a.y) + (a.z + a.w)) + ((b4.x + b4.y) + (b4.z + b4.w)) + (((c.x + c.y) + (c.z + c.w)) + ((d.x + d.y) + (d.z + d.w)));
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    if (half == 0 && row < cnt) out[g0 + row] = acc;
    buf ^= 1;   // the buffer written two rounds ago is free again: every lane passed a __syncwarp after reading it
  }
}

// RAYGRAD (ray-gradient flavour, cfn_flow_composite_bwd_rays): also writes, per (ray, sample), the two sums over k that
// the ray-input gradient needs (cfn_ray_grad_f32): g_zdirect = sum_k gD_k w_k (the depth map's direct z term) and
// g_delta = sum_k dL/d delta_k = sum_k g_alpha_k (1 - alpha_k) softplus(raw sigma_k).  Both are reduced over the 32 lanes
// by a fixed xor butterfly and summed over the latent groups in order; each warp writes only its own samples.  The
// RAYGRAD = false instantiations are the plain K4 kernels.
template <int FT, bool FAST, bool RAYGRAD = false>
__global__ void __launch_bounds__(128, 4)
flow_composite_bwd_kernel(int K, const float* __restrict__ globals, const float* __restrict__ flow_params,
                          const float* __restrict__ z_vals, const float* __restrict__ rays_d, int rays_d_stride,
                          const float* __restrict__ eps_alpha, const float* __restrict__ eps_rgb, int64_t eps_group_rays,
                          int64_t B, int N, int white_bkgd, const float* __restrict__ g_rgb_map,
                          const float* __restrict__ g_depth_map, const float* __restrict__ g_ld,
                          const float* __restrict__ trans,
                          const float* __restrict__ seg_sums, int n_seg,
                          float* __restrict__ g_flow_params, float* __restrict__ g_globals_partial,
                          float* __restrict__ g_zdirect = nullptr, float* __restrict__ g_delta = nullptr) {
  constexpr int F = FT;
  constexpr int PP = 18 * F;
  constexpr int PB = kBwdPB;
  constexpr int NPRE = (PB * PP + 31) / 32;
  extern __shared__ __align__(16) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int zd = (2 * N + 3) & ~3;
  const int per_warp = zd + 2 * PB * PP + 2 * 16 * kBwdGLD;   // every region 16-byte aligned (PB * PP is a multiple of 4)
  float* sz = smem + warp * per_warp;   // z
  float* sd = sz + N;                   // dists * |d|
  float* sP = sz + zd;                  // parameters of the current block [PB][PP]
  float* sO = sP + PB * PP;             // reduced gradient rows of the block [PB][PP]
  float* sG = sO + PB * PP;             // reduction scratch [2][16][GLD]
  // one warp per (ray, sample range): n_seg > 1 splits every ray into n_seg independent back-to-front walks (small
  // batches — the reference trains on 512 rays — would otherwise leave most warp slots of the GPU empty)
  const int64_t wid = (int64_t)blockIdx.x * 4 + warp;
  const int64_t b = wid / n_seg;
  const int seg = (int)(wid % n_seg);
  if (b >= B) return;
  const int seg_len = N / n_seg;
  const int n_lo = seg * seg_len, n_hi = n_lo + seg_len;
  // gradient seeds of the two log-det sums of THIS ray, read from the device (B,2) so that the host never waits for the
  // loss graph and rays of different network calls / loss terms can carry different seeds
  const float gl_a = g_ld[b * 2 + 0];
  const float gl_c = g_ld[b * 2 + 1];
  const int64_t egrp = eps_group_rays > 0 ? b / eps_group_rays : 0;
  eps_alpha += egrp * K;
  eps_rgb += egrp * K * 3;

  for (int n = lane; n < N; n += 32) sz[n] = z_vals[b * N + n];
  const float* d = rays_d + b * rays_d_stride;
  const float dx = d[0], dy = d[1], dz = d[2];
  const float norm = sqrtf(dx * dx + dy * dy + dz * dz);
  __syncwarp();
  for (int n = lane; n < N; n += 32) sd[n] = ((n < N - 1) ? (sz[n + 1] - sz[n]) : 10.0f) * norm;
  __syncwarp();

  const float a_mean = globals[0], a_std = globals[1];
  const float c_mean[3] = {globals[2], globals[3], globals[4]};
  const float c_std[3] = {globals[5], globals[6], globals[7]};
  const float* prow = flow_params + (b * N) * PP;
  float* grow = g_flow_params + (b * N) * PP;
  const float* trow = trans + (b * N) * K;
  const int KG = (K + 31) / 32;
  const int n_blocks = (seg_len + PB - 1) / PB;             // blocks of this warp's range [n_lo, n_hi)
  float gg[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // d/d[a_mean, a_std, c_mean(3), c_std(3)]
  int rbuf = 0;

  for (int kg = 0; kg < KG; ++kg) {
    const int k = kg * 32 + lane;
    const bool active = k < K;
    const float ea = active ? eps_alpha[k] : 0.f;
    float ec[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) ec[c] = active ? eps_rgb[k * 3 + c] : 0.f;
    const float za0 = ea * a_std + a_mean;
    float zc0[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) zc0[c] = ec[c] * c_std[c] + c_mean[c];
    // upstream gradients of this latent sample
    float gC[3] = {0.f, 0.f, 0.f}, gD = 0.f;
    if (active) {
#pragma unroll
      for (int c = 0; c < 3; ++c) gC[c] = g_rgb_map[(b * 3 + c) * K + k];
      if (g_depth_map) gD = g_depth_map[b * K + k];
    }
    const float gA = white_bkgd ? -(gC[0] + gC[1] + gC[2]) : 0.f;
    const float gla = active ? gl_a : 0.f, glc = active ? gl_c : 0.f;

    // suffix sum S = sum over the samples behind this range of v_m w_m: linear in the forward's range sums
    float S = 0.f;
    if (active)
      for (int s2 = seg + 1; s2 < n_seg; ++s2) {
        const float* o = seg_sums + ((b * n_seg + s2) * 5) * K + k;
        S += gC[0] * o[0] + gC[1] * o[K] + gC[2] * o[2 * K] + gD * o[3 * K] + gA * o[4 * K];
      }
    // register prefetch of the next block's parameters (and of the next point's transmittance) while the current one is
    // processed
    float pre[NPRE];
    {
      const int c = n_blocks - 1, n0 = n_lo + c * PB, cnt = (n_hi - n0) * PP;
#pragma unroll
      for (int u = 0; u < NPRE; ++u) pre[u] = (lane + 32 * u < cnt) ? __ldg(prow + (int64_t)n0 * PP + lane + 32 * u) : 0.f;
    }
    float t_next = active ? __ldg(trow + (int64_t)(n_hi - 1) * K + k) : 0.f;
    for (int c = n_blocks - 1; c >= 0; --c) {
      const int n0 = n_lo + c * PB;
      const int npts = min(PB, n_hi - n0);
#pragma unroll
      for (int u = 0; u < NPRE; ++u) if (lane + 32 * u < PB * PP) sP[lane + 32 * u] = pre[u];
      __syncwarp();
      if (c > 0) {
        const int m0 = n0 - PB;   // full block
#pragma unroll
        for (int u = 0; u < NPRE; ++u) pre[u] = (lane + 32 * u < PB * PP) ? __ldg(prow + (int64_t)m0 * PP + lane + 32 * u) : 0.f;
      }
      // NOT unrolled: one point is ~1200 instructions; four copies of the body fell out of the instruction cache (the
      // first capture showed two instruction-fetch stalls per issued instruction, profiles/r02_prof_k2k4_summary.csv)
#pragma unroll 1
      for (int i = npts - 1; i >= 0; --i) {
        {
          const int n = n0 + i;
          const float T = t_next;
          if (n > n_lo) t_next = active ? __ldg(trow + (int64_t)(n - 1) * K + k) : 0.f;
          const float* Pn = sP + i * PP;
          float* On = sO + i * PP;
          // recompute alpha stack with intermediates
          float za_in[F], ta[F];
          float za = za0;
#pragma unroll
          for (int f = 0; f < F; ++f) {
            za_in[f] = za;
            ta[f] = tanh_<FAST>(Pn[F + f] * za + Pn[2 * F + f]);
            za += Pn[f] * ta[f];
          }
          // recompute rgb stack with intermediates
          float zp[F][3], tc[F][3];
          float z[3] = {zc0[0], zc0[1], zc0[2]};
#pragma unroll
          for (int f = 0; f < F; ++f) {
            const float* Q = Pn + 3 * F + kRgbFlowRec * f;
            const bool odd = f & 1;
            zp[f][0] = odd ? z[2] : z[0]; zp[f][1] = z[1]; zp[f][2] = odd ? z[0] : z[2];
            tc[f][0] = tanh_<FAST>(Q[6] * zp[f][0] + Q[7] * zp[f][1] + Q[8] * zp[f][2] + Q[12]);
            tc[f][1] = tanh_<FAST>(Q[9] * zp[f][1] + Q[10] * zp[f][2] + Q[13]);
            tc[f][2] = tanh_<FAST>(Q[11] * zp[f][2] + Q[14]);
            const float s0 = Q[0] * tc[f][0] + Q[1] * tc[f][1] + Q[2] * tc[f][2];
            const float s1 = Q[3] * tc[f][1] + Q[4] * tc[f][2];
            const float s2 = Q[5] * tc[f][2];
            z[0] += odd ? s2 : s0; z[1] += s1; z[2] += odd ? s0 : s2;
          }
          // ---- compositing adjoint (Appendix A.2) ----
          const float sig_za = sigmoid_<FAST>(za);
          const float alpha = 1.0f - exp_<FAST>(-softplus_<FAST>(za) * sd[n]);
          const float w = alpha * T;
          const float q = (1.0f - alpha) + 1e-10f;
          float col[3];
#pragma unroll
          for (int cc = 0; cc < 3; ++cc) col[cc] = sigmoid_<FAST>(z[cc]);
          const float v = gC[0] * col[0] + gC[1] * col[1] + gC[2] * col[2] + gD * sz[n] + gA;
          const float g_alpha = v * T - S / q;
          S += v * w;
          // d alpha / d raw_sigma = (1-alpha) * delta * sigmoid(raw_sigma);  entropy activation term (models.py:263)
          float g_za = g_alpha * (1.0f - alpha) * sd[n] * sig_za + gl_a * (1.0f - sig_za);
          if constexpr (RAYGRAD) {
            // d alpha / d delta = (1 - alpha) * softplus(raw_sigma); inactive lanes contribute exact zeros
            float rz = active ? gD * w : 0.f;
            float rd = active ? g_alpha * (1.0f - alpha) * softplus_<FAST>(za) : 0.f;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              rz += __shfl_xor_sync(0xffffffffu, rz, o);
              rd += __shfl_xor_sync(0xffffffffu, rd, o);
            }
            if (lane == 0) {
              if (kg == 0) { g_zdirect[b * N + n] = rz; g_delta[b * N + n] = rd; }
              else { g_zdirect[b * N + n] += rz; g_delta[b * N + n] += rd; }
            }
          }
          float gz[3];
#pragma unroll
          for (int cc = 0; cc < 3; ++cc)
            gz[cc] = w * gC[cc] * col[cc] * (1.0f - col[cc]) + gl_c * (1.0f - 2.0f * col[cc]);  // models.py:278
          if (!active) { g_za = 0.f; gz[0] = gz[1] = gz[2] = 0.f; }

          // ---- alpha stack adjoint (Appendix A.1 with z_size 1) ----
          float ga[3 * F];
#pragma unroll
          for (int f = F - 1; f >= 0; --f) {
            const float d1 = Pn[f], d2 = Pn[F + f];
            const float t = ta[f], omt2 = 1.0f - t * t;
            const float u = omt2 * (d1 * d2) + 1.0f;
            const float sgn = (u > 0.f) ? 1.f : ((u < 0.f) ? -1.f : 0.f);
            const float sl = gla * sgn / (fabsf(u) + 1e-8f);
            const float g_d1 = g_za * t + sl * omt2 * d2;
            const float gt = d1 * g_za + sl * (-2.0f * t * d1 * d2);
            const float gpre = gt * omt2;
            const float g_d2 = gpre * za_in[f] + sl * omt2 * d1;
            g_za = g_za + d2 * gpre;
            ga[f] = g_d1; ga[F + f] = g_d2; ga[2 * F + f] = gpre;
          }
          reduce_rows_over_lanes<3 * F>(ga, sG, rbuf, On, lane);
          // ---- rgb stack adjoint ----
#pragma unroll
          for (int f = F - 1; f >= 0; --f) {
            const float* Q = Pn + 3 * F + kRgbFlowRec * f;
            float G[kRgbFlowRec];
            const bool odd = f & 1;
            // gy = P g'
            const float gy0 = odd ? gz[2] : gz[0], gy1 = gz[1], gy2 = odd ? gz[0] : gz[2];
            const float t0 = tc[f][0], t1 = tc[f][1], t2 = tc[f][2];
            const float o0 = 1.0f - t0 * t0, o1 = 1.0f - t1 * t1, o2 = 1.0f - t2 * t2;
            const float dd0 = Q[0] * Q[6], dd1 = Q[3] * Q[9], dd2 = Q[5] * Q[11];
            const float u0 = o0 * dd0 + 1.0f, u1 = o1 * dd1 + 1.0f, u2 = o2 * dd2 + 1.0f;
            const float sl0 = glc * ((u0 > 0.f) ? 1.f : ((u0 < 0.f) ? -1.f : 0.f)) / (fabsf(u0) + 1e-8f);
            const float sl1 = glc * ((u1 > 0.f) ? 1.f : ((u1 < 0.f) ? -1.f : 0.f)) / (fabsf(u1) + 1e-8f);
            const float sl2 = glc * ((u2 > 0.f) ? 1.f : ((u2 < 0.f) ? -1.f : 0.f)) / (fabsf(u2) + 1e-8f);
            // gR1 = gy t^T (upper), diagonal gets the log-det term
            G[0] = gy0 * t0 + sl0 * o0 * Q[6];
            G[1] = gy0 * t1;
            G[2] = gy0 * t2;
            G[3] = gy1 * t1 + sl1 * o1 * Q[9];
            G[4] = gy1 * t2;
            G[5] = gy2 * t2 + sl2 * o2 * Q[11];
            // gt = R1^T gy + log-det term
            const float gt0 = Q[0] * gy0 + sl0 * (-2.0f * t0 * dd0);
            const float gt1 = Q[1] * gy0 + Q[3] * gy1 + sl1 * (-2.0f * t1 * dd1);
            const float gt2 = Q[2] * gy0 + Q[4] * gy1 + Q[5] * gy2 + sl2 * (-2.0f * t2 * dd2);
            const float gp0 = gt0 * o0, gp1 = gt1 * o1, gp2 = gt2 * o2;
            // gR2 = gpre zp^T (upper), diagonal gets the log-det term
            G[6] = gp0 * zp[f][0] + sl0 * o0 * Q[0];
            G[7] = gp0 * zp[f][1];
            G[8] = gp0 * zp[f][2];
            G[9] = gp1 * zp[f][1] + sl1 * o1 * Q[3];
            G[10] = gp1 * zp[f][2];
            G[11] = gp2 * zp[f][2] + sl2 * o2 * Q[5];
            G[12] = gp0;
            G[13] = gp1;
            G[14] = gp2;
            // gz = g' + P (R2^T gpre)
            const float r0 = Q[6] * gp0;
            const float r1 = Q[7] * gp0 + Q[9] * gp1;
            const float r2 = Q[8] * gp0 + Q[10] * gp1 + Q[11] * gp2;
            gz[0] += odd ? r2 : r0;
            gz[1] += r1;
            gz[2] += odd ? r0 : r2;
            reduce_rows_over_lanes<kRgbFlowRec>(G, sG, rbuf, On + 3 * F + kRgbFlowRec * f, lane);
          }
          // gradients of the base samples z0 = eps*std + mean
          gg[0] += g_za; gg[1] += ea * g_za;
#pragma unroll
          for (int cc = 0; cc < 3; ++cc) { gg[2 + cc] += gz[cc]; gg[5 + cc] += ec[cc] * gz[cc]; }
        }
      }
      // the block's reduced gradient rows leave as contiguous stores
      __syncwarp();
      {
        float* dst = grow + (int64_t)n0 * PP;
        const int cnt = npts * PP;
        if (kg == 0) { for (int j = lane; j < cnt; j += 32) dst[j] = sO[j]; }
        else { for (int j = lane; j < cnt; j += 32) dst[j] += sO[j]; }
      }
      __syncwarp();
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) gg[j] += __shfl_xor_sync(0xffffffffu, gg[j], o);
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) g_globals_partial[wid * 8 + j] = gg[j];
  }
}

int launch_flow_composite_bwd(int fast_math, int F, int K, const float* globals, const float* flow_params, const float* z_vals,
                              const float* rays_d, int rays_d_stride, const float* eps_alpha, const float* eps_rgb,
                              int64_t eps_group_rays, int64_t B, int N, int white_bkgd, const float* g_rgb_map,
                              const float* g_depth_map, const float* g_ld, const float* trans, const float* seg_sums,
                              int n_seg, float* g_flow_params, float* g_globals_partial, cudaStream_t s,
                              float* g_zdirect, float* g_delta) {
  if (B == 0) return CFN_OK;
  if (!seg_sums || n_seg < 1) n_seg = 1;
  CFN_CHECK_ARG(N % n_seg == 0 && (N / n_seg) >= 1, "flow_composite_bwd: N=%d is not a multiple of n_segments=%d", N, n_seg);
  CFN_CHECK_ARG(F >= 1 && F <= kMaxF, "flow_composite_bwd: n_flows=%d unsupported (1..%d)", F, kMaxF);
  CFN_CHECK_ARG(N >= 2 && N <= 4096 && K >= 1, "flow_composite_bwd: unsupported N=%d (2..4096) K=%d", N, K);
  const int PP = 18 * F;
  size_t smem = (size_t)4 * (((2 * N + 3) & ~3) + 2 * kBwdPB * PP + 2 * 16 * kBwdGLD) * sizeof(float);
  unsigned grid = (unsigned)((B * n_seg + 3) / 4);
#define CFN_BWD_CASE(FF)                                                                                             \
  case FF: {                                                                                                         \
    auto kern = g_zdirect ? (fast_math ? flow_composite_bwd_kernel<FF, true, true> : flow_composite_bwd_kernel<FF, false, true>) \
                          : (fast_math ? flow_composite_bwd_kernel<FF, true> : flow_composite_bwd_kernel<FF, false>);  \
    if (smem > 48 * 1024) CFN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    kern<<<grid, 128, smem, s>>>(K, globals, flow_params, z_vals, rays_d, rays_d_stride, eps_alpha, eps_rgb,         \
                                 eps_group_rays, B, N, white_bkgd, g_rgb_map, g_depth_map, g_ld, trans, seg_sums,    \
                                 n_seg, g_flow_params, g_globals_partial, g_zdirect, g_delta);                       \
  } break;
  switch (F) {
    CFN_BWD_CASE(1) CFN_BWD_CASE(2) CFN_BWD_CASE(3) CFN_BWD_CASE(4) CFN_BWD_CASE(5) CFN_BWD_CASE(6) CFN_BWD_CASE(7)
    CFN_BWD_CASE(8)
  }
#undef CFN_BWD_CASE
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

}  // namespace cfn
