// F5 evaluation: per-pixel uncertainty records and the sparsification curves / AUSE of V views of P pixels each.
//
// Records (eval_records_kernel, one warp per ray): from the K-reduction (kstats of K2) and the trainer-loss partials (F1)
// of the same maps, u = mean_c s_c^2, e = partial[1] / 3, a = mean_c |mu_c - t_c|, nll = partial[0] / 3; with depth
// targets also the unbiased variance of depth over k, and the squared / absolute error of its mean.
//
// Sparsification (DESIGN §5, F5): three device-wide radix sorts over composite 64-bit keys (view << 32 | float bits; the
// bits of a non-negative float sort in value order, the view keeps the views apart in one sort):
//   1. u with the flat pixel index as payload (stable: ties keep the lower pixel first), then e and a gathered in that
//      order;  2. e, keys only;  3. a, keys only.
// That gives four sorted sequences per view: [e by u, e ascending, a by u, a ascending].  sparsify_bins_kernel sums the
// disjoint ranges [m_{i+1}, m_i) of each in fp64 (one block per bin, fixed-order reduction), so every element is read
// once; sparsify_finalize_kernel takes the suffix sums of the S bins, writes the normalised curves and the AUSE.  The
// result is bitwise deterministic and, per view, independent of the other views of the call.
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace cfn {

namespace {

constexpr int kBinThreads = 256;

__device__ __forceinline__ float warp_sum_f(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ int64_t keep_count(int64_t P, int S, int i) {   // m_i = P - floor(i P / S), m_S = 0
  return P - (i * P) / S;
}

// bits of a non-negative float (the sign of -0.0 dropped) under the view index
__device__ __forceinline__ unsigned long long view_key(int64_t view, float x) {
  return ((unsigned long long)view << 32) | (unsigned long long)(__float_as_uint(x) & 0x7fffffffu);
}

}  // namespace

__global__ void eval_records_kernel(const float* __restrict__ kstats, const float* __restrict__ partial,
                                    const float* __restrict__ target_rgb, const float* __restrict__ depth_map,
                                    const float* __restrict__ target_depth, int64_t B, int K, float* __restrict__ u,
                                    float* __restrict__ sq_err, float* __restrict__ abs_err, float* __restrict__ nll,
                                    float* __restrict__ depth_u, float* __restrict__ depth_sq_err,
                                    float* __restrict__ depth_abs_err) {
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  if (lane == 0) {
    const float* ks = kstats + b * 8;
    const float* t = target_rgb + b * 3;
    u[b] = (ks[3] * ks[3] + ks[4] * ks[4] + ks[5] * ks[5]) / 3.0f;
    abs_err[b] = (fabsf(ks[0] - t[0]) + fabsf(ks[1] - t[1]) + fabsf(ks[2] - t[2])) / 3.0f;
    sq_err[b] = partial[b * 3 + 1] / 3.0f;
    nll[b] = partial[b * 3 + 0] / 3.0f;
  }
  if (depth_map) {
    const float* d = depth_map + b * K;
    float s = 0.f;
    for (int k = lane; k < K; k += 32) s += d[k];
    const float mean = warp_sum_f(s) / (float)K;
    float q = 0.f;
    for (int k = lane; k < K; k += 32) q += (d[k] - mean) * (d[k] - mean);
    q = warp_sum_f(q);
    if (lane == 0) {
      const float err = mean - target_depth[b];
      depth_u[b] = q / (float)(K - 1);
      depth_sq_err[b] = err * err;
      depth_abs_err[b] = fabsf(err);
    }
  }
}

__global__ void sparsify_keys_kernel(const float* __restrict__ x, int64_t P, int64_t n, unsigned long long* __restrict__ keys,
                                     int* __restrict__ index) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  keys[j] = view_key(j / P, x[j]);
  if (index) index[j] = (int)j;
}

__global__ void sparsify_gather_kernel(const int* __restrict__ order, const float* __restrict__ e, const float* __restrict__ a,
                                       int64_t n, float* __restrict__ e_by_u, float* __restrict__ a_by_u) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int src = order[j];
  e_by_u[j] = e[src];
  a_by_u[j] = a[src];
}

// grid (S, V, 4): bin i of view v and sequence q = sum over [m_{i+1}, m_i) in fp64.  q = 0 / 2: e / a in the order of
// ascending u (floats); q = 1 / 3: e / a sorted (the float bits are the low half of the sorted keys).
__global__ void __launch_bounds__(kBinThreads) sparsify_bins_kernel(const float* __restrict__ e_by_u,
                                                                     const float* __restrict__ a_by_u,
                                                                     const unsigned long long* __restrict__ e_sorted,
                                                                     const unsigned long long* __restrict__ a_sorted,
                                                                     int64_t P, int S, double* __restrict__ bins) {
  __shared__ double red[kBinThreads / 32];
  const int i = blockIdx.x, v = blockIdx.y, q = blockIdx.z;
  const int64_t lo = keep_count(P, S, i + 1), hi = keep_count(P, S, i);
  const int64_t base = (int64_t)v * P;
  double s = 0.0;
  if (q == 0 || q == 2) {
    const float* x = (q == 0 ? e_by_u : a_by_u) + base;
    for (int64_t j = lo + threadIdx.x; j < hi; j += kBinThreads) s += (double)x[j];
  } else {
    const unsigned long long* x = (q == 1 ? e_sorted : a_sorted) + base;
    for (int64_t j = lo + threadIdx.x; j < hi; j += kBinThreads) s += (double)__uint_as_float((unsigned)x[j]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kBinThreads / 32; ++w) t += red[w];
    bins[((int64_t)v * 4 + q) * S + i] = t;
  }
}

// one thread per (view, metric): metric 0 = RMSE (sequences 0 / 1), 1 = MAE (sequences 2 / 3).  The prefix sum over
// the kept pixels at fraction i is the suffix sum of bins i..S-1; each curve is divided by its own value at i = 0.
__global__ void sparsify_finalize_kernel(const double* __restrict__ bins, int64_t V, int64_t P, int S,
                                         float* __restrict__ curves, float* __restrict__ ause) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= V * 2) return;
  const int64_t v = t >> 1;
  const int metric = (int)(t & 1);
  const double* bc = bins + ((int64_t)v * 4 + 2 * metric) * S;     // the curve ordered by u
  const double* bo = bc + S;                                        // its oracle
  const bool root = metric == 0;
  double tc = 0.0, to = 0.0;
  for (int i = S - 1; i >= 0; --i) { tc += bc[i]; to += bo[i]; }
  const double n0 = (double)P;
  const double c0 = root ? sqrt(tc / n0) : tc / n0, o0 = root ? sqrt(to / n0) : to / n0;
  float* out_c = curves + ((int64_t)v * 4 + 2 * metric) * S;
  float* out_o = out_c + S;
  double sc = 0.0, so = 0.0, area = 0.0, d_next = 0.0;
  for (int i = S - 1; i >= 0; --i) {
    sc += bc[i];
    so += bo[i];
    const double m = (double)keep_count(P, S, i);
    double c = root ? sqrt(sc / m) : sc / m, o = root ? sqrt(so / m) : so / m;
    c = c0 > 0.0 ? c / c0 : 0.0;
    o = o0 > 0.0 ? o / o0 : 0.0;
    out_c[i] = (float)c;
    out_o[i] = (float)o;
    const double d = c - o;
    if (i < S - 1) area += (d + d_next) * 0.5 / (double)S;
    d_next = d;
  }
  ause[v * 2 + metric] = (float)area;
}

namespace {

struct SparsifyLayout {
  size_t keys_in, keys_u, keys_a, index_in, index_u, e_by_u, a_by_u, bins, cub_tmp, cub_bytes, total;
};

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

int end_bit_for(int64_t V) {
  int b = 0;
  while (((int64_t)1 << b) < V) ++b;
  return 32 + b;
}

int sparsify_layout(int64_t V, int64_t P, int S, SparsifyLayout* L) {
  const int64_t n = V * P;
  const int eb = end_bit_for(V);
  size_t pairs = 0, keys = 0;
  CFN_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, pairs, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                           (const int*)nullptr, (int*)nullptr, (int)n, 0, eb, (cudaStream_t)0));
  CFN_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, keys, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                          (int)n, 0, eb, (cudaStream_t)0));
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += align256(bytes); return o; };
  L->keys_in = take(n * sizeof(unsigned long long));
  L->keys_u = take(n * sizeof(unsigned long long));      // sort 1's keys, then sort 2's output (e ascending)
  L->keys_a = take(n * sizeof(unsigned long long));      // sort 3's output (a ascending)
  L->index_in = take(n * sizeof(int));
  L->index_u = take(n * sizeof(int));
  L->e_by_u = take(n * sizeof(float));
  L->a_by_u = take(n * sizeof(float));
  L->bins = take((size_t)V * 4 * S * sizeof(double));
  L->cub_bytes = pairs > keys ? pairs : keys;
  L->cub_tmp = take(L->cub_bytes);
  L->total = off + 256;                                   // the caller's base need not be 256-byte aligned
  return CFN_OK;
}

}  // namespace

int sparsify_workspace_bytes(int64_t V, int64_t P, int S, size_t* out) {
  SparsifyLayout L;
  const int rc = sparsify_layout(V, P, S, &L);
  if (rc != CFN_OK) return rc;
  *out = L.total;
  return CFN_OK;
}

int launch_eval_records(const float* kstats, const float* partial, const float* target_rgb, const float* depth_map,
                        const float* target_depth, int64_t B, int K, float* u, float* sq_err, float* abs_err, float* nll,
                        float* depth_u, float* depth_sq_err, float* depth_abs_err, cudaStream_t s) {
  if (B == 0) return CFN_OK;
  const int64_t threads = B * 32;
  eval_records_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(kstats, partial, target_rgb, depth_map, target_depth,
                                                                        B, K, u, sq_err, abs_err, nll, depth_u, depth_sq_err,
                                                                        depth_abs_err);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

int launch_sparsify(const float* u, const float* e, const float* a, int64_t V, int64_t P, int S, void* workspace,
                    size_t workspace_bytes, float* curves, float* ause, cudaStream_t s) {
  SparsifyLayout L;
  int rc = sparsify_layout(V, P, S, &L);
  if (rc != CFN_OK) return rc;
  if (workspace_bytes < L.total) {
    set_error("cfn_sparsification_f32: workspace %zu bytes < required %zu", workspace_bytes, L.total);
    return CFN_ENOMEM;
  }
  char* w = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  auto* keys_in = (unsigned long long*)(w + L.keys_in);
  auto* keys_u = (unsigned long long*)(w + L.keys_u);
  auto* keys_a = (unsigned long long*)(w + L.keys_a);
  auto* index_in = (int*)(w + L.index_in);
  auto* index_u = (int*)(w + L.index_u);
  auto* e_by_u = (float*)(w + L.e_by_u);
  auto* a_by_u = (float*)(w + L.a_by_u);
  auto* bins = (double*)(w + L.bins);
  void* tmp = w + L.cub_tmp;
  const int64_t n = V * P;
  const int eb = end_bit_for(V);
  const unsigned grid = (unsigned)((n + 255) / 256);
  size_t tb = L.cub_bytes;

  sparsify_keys_kernel<<<grid, 256, 0, s>>>(u, P, n, keys_in, index_in);
  CFN_LAUNCH_CHECK();
  CFN_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, keys_in, keys_u, index_in, index_u, (int)n, 0, eb, s));
  sparsify_gather_kernel<<<grid, 256, 0, s>>>(index_u, e, a, n, e_by_u, a_by_u);
  CFN_LAUNCH_CHECK();
  sparsify_keys_kernel<<<grid, 256, 0, s>>>(e, P, n, keys_in, nullptr);
  CFN_LAUNCH_CHECK();
  tb = L.cub_bytes;
  CFN_CUDA(cub::DeviceRadixSort::SortKeys(tmp, tb, keys_in, keys_u, (int)n, 0, eb, s));
  sparsify_keys_kernel<<<grid, 256, 0, s>>>(a, P, n, keys_in, nullptr);
  CFN_LAUNCH_CHECK();
  tb = L.cub_bytes;
  CFN_CUDA(cub::DeviceRadixSort::SortKeys(tmp, tb, keys_in, keys_a, (int)n, 0, eb, s));
  sparsify_bins_kernel<<<dim3((unsigned)S, (unsigned)V, 4), kBinThreads, 0, s>>>(e_by_u, a_by_u, keys_u, keys_a, P, S, bins);
  CFN_LAUNCH_CHECK();
  sparsify_finalize_kernel<<<(unsigned)((V * 2 + 63) / 64), 64, 0, s>>>(bins, V, P, S, curves, ause);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

}  // namespace cfn
