// The layer-by-layer network stage (K5): positional encoding (run_nerf_helpers.py:21-69), the 8x512 trunk with skip-concat,
// the conditioning heads (model/models.py:165-186) and the amortised flow parameters (models.py:358-385, done ONCE
// per point instead of K times), forward with optional saved activations and the full backward (dgrad chain +
// split-K wgrad).  The contractions run as fp32 CUDA-core FMAs (sgemm.cu) in CFN_PREC_FP32 — the 1e-5 "check" mode
// — and as TMA-fed tcgen05 kind::tf32 GEMMs (gemm_tc.cu) in every other mode: that is the training path of the
// bf16 / fp16 modes and the whole network stage of CFN_PREC_TF32.  In the tensor-core flavour every buffer that is a
// later GEMM's operand (activations, gradients, weights) is stored ROUNDED to tf32, because the tensor core truncates.
#include <cuda_bf16.h>

#include <algorithm>

#include "handle.h"

namespace cfn {

// ---------------------------------------------------------------------------------------------------
// workspace layout (floats; M = number of points)
// ---------------------------------------------------------------------------------------------------
// Buffers that hold activations / gradients are addressed in ELEMENTS (fp32, or bf16 when h->chain_bf16) through
// float* bases: `at(base, n)` advances by n elements (n is always a multiple of 8 in bf16 mode), region sizes are in
// 4-byte slots.
struct ChainLayout {
  int ld5, ldv, ldg;
  int gpa, ldGP;                            // gradient of the flow record: [3F | pad to 8 | 15F | pad to 8]
  int64_t X5, V, H, v, ha, hr;            // forward
  int64_t P, GP, G1, G2, gv, gh, dAm, dWp;  // saved outputs / backward scratch
  int64_t MB, mbv; int bw, bwv;             // ReLU bit masks of the trunk layers / the view layer (words per row)
  int nH;
  int64_t total;
};

// the tensor-core engine carries relu'(h) from the forward to the dgrad GEMMs as bit masks (needs every ReLU layer on it)
static bool use_bits(const CfnHandle* h) { return h->gemm_tc && h->cfg.W % 8 == 0; }

static ChainLayout make_layout(const CfnHandle* h, int64_t M, int save) {
  ChainLayout L;
  const int W = h->cfg.W;
  L.ld5 = h->gp + W;          // [gamma(p) | pad to 4 | h]: the h columns start 16-byte aligned
  L.ldv = W + h->gd;          // [feature | gamma(d) | pad to 4]
  L.ldg = L.ld5 > L.ldv ? L.ld5 : L.ldv;
  const int wc = W + ((h->cfg.h_alpha + 7) & ~7);   // [g_feat | g_h_alpha] rows of the fused head dgrad
  if (wc > L.ldg) L.ldg = wc;
  L.gpa = (3 * h->cfg.F + 7) & ~7;
  L.ldGP = L.gpa + ((15 * h->cfg.F + 7) & ~7);
  L.nH = save ? h->cfg.D : 2;
  const int e = h->chain_bf16 ? 2 : 1;              // elements per 4-byte slot
  int64_t o = 0;
  auto take = [&](int64_t n) { int64_t r = o; o += (n + 3) & ~(int64_t)3; return r; };   // n 4-byte slots
  auto take_e = [&](int64_t n) { return take((n + e - 1) / e); };                        // n elements
  L.X5 = take_e(M * L.ld5);
  L.V = take_e(M * L.ldv);
  L.H = take_e((int64_t)L.nH * M * W);
  L.v = take_e(M * (W / 2));
  L.ha = take_e(M * h->cfg.h_alpha);
  L.hr = take_e(M * h->cfg.h_rgb);
  L.P = L.GP = L.G1 = L.G2 = L.gv = L.gh = L.dAm = L.dWp = L.MB = L.mbv = 0;
  L.bw = (W + 31) / 32; L.bwv = (W / 2 + 31) / 32;
  if (save) {
    L.P = take(M * h->PP);
    L.GP = take_e(M * L.ldGP);
    L.G1 = take_e(M * L.ldg);
    L.G2 = take_e(M * L.ldg);
    L.gv = take_e(M * (W / 2));
    int hm = h->cfg.h_alpha > h->cfg.h_rgb ? h->cfg.h_alpha : h->cfg.h_rgb;
    L.gh = take_e(M * hm);
    L.dAm = take((int64_t)h->PP * (hm + 1));
    L.dWp = take((int64_t)W * (h->gp + W + 4));   // padded weight gradient of the odd-width layers
    if (use_bits(h)) {
      L.MB = take((int64_t)h->cfg.D * M * L.bw);
      L.mbv = take(M * L.bwv);
    }
  }
  L.total = o;
  return L;
}

static inline float* at(const CfnHandle* h, float* base, int64_t elems) { return base + (h->chain_bf16 ? elems / 2 : elems); }
static inline const float* at(const CfnHandle* h, const float* base, int64_t elems) { return base + (h->chain_bf16 ? elems / 2 : elems); }

size_t chain_workspace_floats(const CfnHandle* h, int64_t M, int save) {
  return (size_t)make_layout(h, M, save).total;
}

// ---------------------------------------------------------------------------------------------------
// positional encoding: gamma(p) -> X5[:, 0:in_pos], gamma(d) -> V[:, W:W+in_dir]
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void embed3(float x, float y, float z, int L, float* out) {
  out[0] = x; out[1] = y; out[2] = z;
  float f = 1.0f;
  for (int l = 0; l < L; ++l) {
    float* o = out + 3 + 6 * l;
    const float xf = x * f, yf = y * f, zf = z * f;   // exact: f is a power of two (helpers:38)
    o[0] = sinf(xf); o[1] = sinf(yf); o[2] = sinf(zf);
    o[3] = cosf(xf); o[4] = cosf(yf); o[5] = cosf(zf);
    f *= 2.0f;
  }
}

__device__ __forceinline__ float round_tf32(float x) {
  uint32_t r; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x)); return __uint_as_float(r);
}

// element store of an operand buffer: mode 0 = fp32 as is, 1 = fp32 rounded to tf32, 2 = bf16
__device__ __forceinline__ void store_elem(float* base, int64_t idx, float v, int mode) {
  if (mode == 2) reinterpret_cast<__nv_bfloat16*>(base)[idx] = __float2bfloat16_rn(v);
  else base[idx] = (mode == 1) ? round_tf32(v) : v;
}

// n_pos / n_dir: padded widths (pad columns are written as zeros); round: store tf32-rounded values.
// One thread encodes one point into shared memory; the block then writes the rows out with consecutive lanes on
// consecutive columns (the rows are 2304 bytes apart in X5: per-thread row stores would touch 32 lines per instruction).
constexpr int ENC_PTS = 128, ENC_MAXW = 104;   // up to multires 16: 3 + 6*16 = 99 (+ pad)
__global__ void __launch_bounds__(ENC_PTS)
encode_kernel(const float* __restrict__ rays, const float* __restrict__ z_vals, const float* __restrict__ pts,
              const float* __restrict__ viewdirs, int64_t M, int N, int L_pos, int L_dir, float* __restrict__ X5, int ld5,
              float* __restrict__ Vd, int ldv, int n_pos, int n_dir, int mode) {
  extern __shared__ float enc_smem[];
  const int lp = n_pos | 1, ldd = n_dir | 1;            // odd row strides: conflict-free per-thread rows
  float* sp = enc_smem;
  float* sd = enc_smem + ENC_PTS * lp;
  const int64_t m0 = (int64_t)blockIdx.x * ENC_PTS;
  const int64_t m = m0 + threadIdx.x;
  if (m < M) {
    const int64_t b = m / N;
    float px, py, pz;
    if (pts) {
      px = pts[m * 3 + 0]; py = pts[m * 3 + 1]; pz = pts[m * 3 + 2];
    } else {
      const float* r = rays + b * 11;
      const float z = z_vals[m];
      // pts = rays_o + rays_d * z (main:534): separate multiply and add, as torch evaluates it
      px = __fadd_rn(r[0], __fmul_rn(r[3], z));
      py = __fadd_rn(r[1], __fmul_rn(r[4], z));
      pz = __fadd_rn(r[2], __fmul_rn(r[5], z));
    }
    float* rp = sp + threadIdx.x * lp;
    float* rd = sd + threadIdx.x * ldd;
    embed3(px, py, pz, L_pos, rp);
    const float* vd = viewdirs ? (viewdirs + b * 3) : (rays + b * 11 + 8);
    embed3(vd[0], vd[1], vd[2], L_dir, rd);
    for (int c = 3 + 6 * L_pos; c < n_pos; ++c) rp[c] = 0.f;
    for (int c = 3 + 6 * L_dir; c < n_dir; ++c) rd[c] = 0.f;
  }
  __syncthreads();
  const int rows = (int)min((int64_t)ENC_PTS, M - m0);
  for (int i = threadIdx.x; i < rows * n_pos; i += ENC_PTS) {
    const int r = i / n_pos, c = i - r * n_pos;
    const float v = sp[r * lp + c];
    store_elem(X5, (m0 + r) * ld5 + c, v, mode);
  }
  for (int i = threadIdx.x; i < rows * n_dir; i += ENC_PTS) {
    const int r = i / n_dir, c = i - r * n_dir;
    const float v = sd[r * ldd + c];
    store_elem(Vd, (m0 + r) * ldv + c, v, mode);
  }
}

// operand copy of every weight matrix: padded row stride, gap after gamma(p) in the skip layer, optional tf32 rounding
struct RepackTable {
  int64_t src[64], dst[64];
  int rows[64], cols[64], ld[64], gap_at[64], gap[64];
  int n;
};
__global__ void repack_weights_kernel(const float* __restrict__ w32, float* __restrict__ wg, RepackTable t, int mode) {
  const int s = blockIdx.y;
  const int64_t n = (int64_t)t.rows[s] * t.cols[s];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / t.cols[s]), c = (int)(i % t.cols[s]);
    const float v = w32[t.src[s] + i];
    // dst is in 4-byte slots: an element index in the buffer's own type
    store_elem(wg, t.dst[s] * (mode == 2 ? 2 : 1) + (int64_t)r * t.ld[s] + c + (c >= t.gap_at[s] ? t.gap[s] : 0), v, mode);
  }
}
__global__ void round_copy_kernel(const float* __restrict__ src, float* __restrict__ dst, int n, int mode) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) store_elem(dst, i, src[i], mode);
}

// ---------------------------------------------------------------------------------------------------
// parameter packing (fp32): flat copy + gathered conditioning matrices
// ---------------------------------------------------------------------------------------------------
struct SlotTable {
  int64_t offset[64];
  int cols[64];
};

__global__ void gather_rows_kernel(const float* __restrict__ w32, SlotTable t, const int* __restrict__ gather, int rows,
                                   int cols, float* __restrict__ out_w, float* __restrict__ out_b) {
  int r = blockIdx.x;
  if (r >= rows) return;
  const int slot_w = gather[r * 4 + 0], slot_b = gather[r * 4 + 1], row = gather[r * 4 + 2];
  for (int c = threadIdx.x; c < cols; c += blockDim.x) out_w[r * cols + c] = w32[t.offset[slot_w] + (int64_t)row * cols + c];
  if (threadIdx.x == 0) out_b[r] = w32[t.offset[slot_b] + row];
}

static SlotTable slot_table(const CfnHandle* h) {
  SlotTable t;
  for (size_t i = 0; i < h->slots.size() && i < 64; ++i) {
    t.offset[i] = h->slots[i].offset;
    t.cols[i] = h->slots[i].cols;
  }
  return t;
}

int pack_fp32(CfnHandle* h, const float* const* params, cudaStream_t s) {
  CFN_CHECK_ARG(h->slots.size() <= 64, "too many parameter tensors");
  // parameters that already sit back to back in slot order (cfnerf_b200.dist.FusedTrainStep flattens them) travel in
  // one copy instead of one per tensor
  bool flat = true;
  for (size_t i = 0; i < h->slots.size(); ++i) flat = flat && (params[i] == params[0] + h->slots[i].offset);
  if (flat) {
    CFN_CUDA(cudaMemcpyAsync(h->w32, params[0], h->n_floats * sizeof(float), cudaMemcpyDeviceToDevice, s));
  } else {
    for (size_t i = 0; i < h->slots.size(); ++i)
      CFN_CUDA(cudaMemcpyAsync(h->w32 + h->slots[i].offset, params[i], h->slots[i].numel * sizeof(float),
                               cudaMemcpyDeviceToDevice, s));
  }
  SlotTable t = slot_table(h);
  gather_rows_kernel<<<3 * h->cfg.F, 64, 0, s>>>(h->w32, t, h->gatherA_dev, 3 * h->cfg.F, h->cfg.h_alpha, h->amA,
                                                 h->amA_b);
  gather_rows_kernel<<<15 * h->cfg.F, 64, 0, s>>>(h->w32, t, h->gatherC_dev, 15 * h->cfg.F, h->cfg.h_rgb, h->amC,
                                                  h->amC_b);
  {
    RepackTable rt;
    rt.n = 0;
    for (size_t i = 0; i < h->slots.size(); ++i) {
      if (!h->wv[i].ld) continue;
      const int k = rt.n++;
      rt.src[k] = h->slots[i].offset; rt.dst[k] = h->wg_offset[i];
      rt.rows[k] = h->slots[i].rows; rt.cols[k] = h->slots[i].cols;
      rt.ld[k] = h->wv[i].ld; rt.gap_at[k] = h->wv[i].gap_at; rt.gap[k] = h->wv[i].gap;
    }
    const int mode = h->chain_bf16 ? 2 : (h->gemm_tc ? 1 : 0);
    repack_weights_kernel<<<dim3(64, rt.n), 256, 0, s>>>(h->w32, h->wg, rt, mode);
    if (h->gemm_tc) {
      const int na = 3 * h->cfg.F * h->cfg.h_alpha, nc = 15 * h->cfg.F * h->cfg.h_rgb;
      round_copy_kernel<<<(na + 255) / 256, 256, 0, s>>>(h->amA, h->amA_g, na, mode);
      round_copy_kernel<<<(nc + 255) / 256, 256, 0, s>>>(h->amC, h->amC_g, nc, mode);
    }
  }
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

// the contraction engine of this handle
static int gemm(const CfnHandle* h, const GemmArgs& g, int round_out, cudaStream_t s) {
  if (g.ab_bf16) {
    CFN_CHECK_ARG(tgemm_supported(g), "bf16 chain: GEMM flavour not available (M %lld N %d K %lld epilogue %d split %d)",
                  (long long)g.M, g.N, (long long)g.K, g.epilogue, g.split_k);
    return launch_tgemm(g, 0, s);
  }
  if (h->gemm_tc && tgemm_supported(g)) return launch_tgemm(g, round_out, s);
  return launch_sgemm(g, s);   // fp32 mode, or a shape the TMA path cannot address (e.g. an odd flow-record width)
}

// ---------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------
static inline const float* Wp(const CfnHandle* h, int slot) { return h->w32 + h->slots[slot].offset; }

// Y(M x out) = epi(X(M x in) W^T + b) for an nn.Linear stored (out, in) row-major
static int linear_fwd(const CfnHandle* h, int slot, const float* X, int64_t ldx, float* Y, int64_t ldy, int64_t M,
                      int epi, const float* aux, cudaStream_t s, uint32_t* mask_out = nullptr, int bits_ld = 0,
                      int round_out = 1) {
  const ParamSlot& w = h->slots[slot];
  const WView& v = h->wv[slot];
  GemmArgs g{};
  g.A = X; g.a_rs = ldx; g.a_cs = 1;
  g.B = v.p; g.b_rs = 1; g.b_cs = v.ld;                // B(k,n) = W[n*ld + k]; pad columns meet zero activations
  g.C = Y; g.c_rs = ldy;
  g.bias = Wp(h, slot + 1);
  g.aux = aux; g.aux_rs = 0;
  g.M = M; g.N = w.rows; g.K = v.ld;
  g.epilogue = epi; g.accumulate = 0; g.split_k = 1;
  g.mask_out = mask_out; g.bits_ld = bits_ld;
  g.ab_bf16 = g.c_bf16 = h->chain_bf16;
  if (mask_out) CFN_CHECK_ARG(tgemm_supported(g), "linear_fwd: ReLU bit masks need the tensor-core engine");
  return gemm(h, g, round_out, s);
}

struct LayerIO {
  const float* in; int64_t ld_in;
  float* out; int64_t ld_out;
};

static LayerIO trunk_io(const CfnHandle* h, const ChainLayout& L, float* ws, int64_t M, int i, int save) {
  const int W = h->cfg.W;
  auto Hbuf = [&](int j) { return at(h, ws + L.H, (int64_t)(save ? j : (j & 1)) * M * W); };
  LayerIO io;
  if (i == 0) { io.in = ws + L.X5; io.ld_in = L.ld5; }
  else if (h->skip >= 0 && i == h->skip + 1) { io.in = ws + L.X5; io.ld_in = L.ld5; }
  else { io.in = Hbuf(i - 1); io.ld_in = W; }
  if (h->skip >= 0 && i == h->skip) { io.out = at(h, ws + L.X5, h->gp); io.ld_out = L.ld5; }
  else { io.out = Hbuf(i); io.ld_out = W; }
  return io;
}

int chain_network_fwd(CfnHandle* h, const float* rays, const float* z_vals, const float* pts, const float* viewdirs,
                     int64_t B, int N, float* flow_params, float* ws, int save, cudaStream_t s) {
  const int64_t M = B * N;
  const int W = h->cfg.W, D = h->cfg.D, F = h->cfg.F;
  ChainLayout L = make_layout(h, M, save);
  const size_t enc_smem = (size_t)ENC_PTS * ((h->gp | 1) + (h->gd | 1)) * sizeof(float);
  static PerDeviceOnce enc_attr;   // function attributes are per device
  if (!enc_attr.done()) {
    CFN_CUDA(cudaFuncSetAttribute((const void*)encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * ENC_PTS * ENC_MAXW * 4));
    enc_attr.mark();
  }
  encode_kernel<<<(unsigned)((M + ENC_PTS - 1) / ENC_PTS), ENC_PTS, enc_smem, s>>>(
      rays, z_vals, pts, viewdirs, M, N, h->cfg.L_pos, h->cfg.L_dir, ws + L.X5, L.ld5, at(h, ws + L.V, W), L.ldv, h->gp, h->gd,
      h->chain_bf16 ? 2 : (h->gemm_tc ? 1 : 0));
  CFN_LAUNCH_CHECK();
  int rc;
  LayerIO last{};
  for (int i = 0; i < D; ++i) {
    LayerIO io = trunk_io(h, L, ws, M, i, save);
    uint32_t* mb = (save && use_bits(h)) ? reinterpret_cast<uint32_t*>(ws + L.MB) + (int64_t)i * M * L.bw : nullptr;
    if ((rc = linear_fwd(h, h->s_pts(i, 0), io.in, io.ld_in, io.out, io.ld_out, M, EPI_RELU, nullptr, s, mb, L.bw))) return rc;
    last = io;
  }
  const float* h7 = last.out;
  const int64_t ld7 = last.ld_out;
  // heads (models.py:175-182)
  // In the fp32-storage tensor-core chain (tf32) the conditioning vectors h_alpha / h_rgb keep their fp32 accumulator
  // value and the two amortisation GEMMs below (N = 3F / 15F, K = 64: 0.2 % of the flops) run on the CUDA cores with the
  // exact fp32 weights: trained-like ("stressed") heads amplify every rounding in front of the flows ~30x, and rounding
  // h and the amortisation weights to tf32 as well took the render outside the 2e-3 bar there (2.8e-3 / 3.9e-3 on
  // predictive mean / std; 1.0e-3 / 1.4e-3 without, the same as the fused fp16 kernel that composes the two matrices).
  const bool exact_amor = h->gemm_tc && !h->chain_bf16;
  const int round_h = exact_amor ? 0 : 1;
  if ((rc = linear_fwd(h, h->s_halpha, h7, ld7, ws + L.ha, h->cfg.h_alpha, M, EPI_NONE, nullptr, s, nullptr, 0, round_h))) return rc;
  if ((rc = linear_fwd(h, h->s_feat, h7, ld7, ws + L.V, L.ldv, M, EPI_NONE, nullptr, s))) return rc;
  if ((rc = linear_fwd(h, h->s_views, ws + L.V, L.ldv, ws + L.v, W / 2, M, EPI_RELU, nullptr, s,
                       (save && use_bits(h)) ? reinterpret_cast<uint32_t*>(ws + L.mbv) : nullptr, L.bwv))) return rc;
  if ((rc = linear_fwd(h, h->s_hrgb, ws + L.v, W / 2, ws + L.hr, h->cfg.h_rgb, M, EPI_NONE, nullptr, s, nullptr, 0, round_h))) return rc;
  // amortised flow parameters, once per point (models.py:358-385)
  {
    GemmArgs g{};
    g.A = ws + L.ha; g.a_rs = h->cfg.h_alpha; g.a_cs = 1;
    g.B = h->amA_g; g.b_rs = 1; g.b_cs = h->cfg.h_alpha;
    g.C = flow_params; g.c_rs = h->PP;
    g.bias = h->amA_b; g.aux = h->tanh_flags; g.aux_rs = 0;
    g.ab_bf16 = h->chain_bf16; g.c_bf16 = 0;       // the flow records stay fp32
    g.M = M; g.N = 3 * F; g.K = h->cfg.h_alpha; g.epilogue = EPI_TANH_MASK; g.split_k = 1;
    if (exact_amor) g.B = h->amA;
    if ((rc = exact_amor ? launch_sgemm(g, s) : gemm(h, g, 0, s))) return rc;
    g.A = ws + L.hr; g.a_rs = h->cfg.h_rgb;
    g.B = exact_amor ? h->amC : h->amC_g; g.b_cs = h->cfg.h_rgb;
    g.C = flow_params + 3 * F;
    g.bias = h->amC_b; g.aux = h->tanh_flags + 3 * F;
    g.N = 15 * F; g.K = h->cfg.h_rgb;
    if ((rc = exact_amor ? launch_sgemm(g, s) : gemm(h, g, 0, s))) return rc;
  }
  if (save) CFN_CUDA(cudaMemcpyAsync(ws + L.P, flow_params, (size_t)M * h->PP * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return CFN_OK;
}

// ---------------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------------
__global__ void tanh_bwd_kernel(const float* __restrict__ g, const float* __restrict__ p, const float* __restrict__ flags,
                                float* __restrict__ out, int64_t total, int PP, int n_alpha, int gpa, int ldGP, int mode) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const float pv = p[i];
  const int c = (int)(i % PP);
  const float v = flags[c] != 0.f ? g[i] * (1.0f - pv * pv) : g[i];
  // record column c -> [alpha block | pad | rgb block] so that both blocks start 16-byte aligned in either storage type
  store_elem(out, (i / PP) * ldGP + (c < n_alpha ? c : gpa + c - n_alpha), v, mode);
}

// out[n] += sum over a slab of rows of g[m*ld + n]   (out pre-zeroed)
__global__ void colsum_kernel(const float* __restrict__ g, int64_t ld, int64_t M, int N, float* __restrict__ out,
                              int rows_per_block) {
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = min(M, r0 + rows_per_block);
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    float s = 0.f;
    for (int64_t m = r0; m < r1; ++m) s += g[m * ld + n];
    atomicAdd(out + n, s);
  }
}

// deterministic variant: 32 columns x 8 row lanes per block, every thread adds its rows in order, the 8 lanes are joined
// in a fixed order (no atomics)
__global__ void colsum_det_kernel(const float* __restrict__ g, int64_t ld, int64_t M, int N, float* __restrict__ out) {
  __shared__ float red[8][32];
  const int c = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + c;
  float s = 0.f;
  if (n < N) for (int64_t m = rl; m < M; m += 8) s += g[m * ld + n];
  red[rl][c] = s;
  __syncthreads();
  if (rl == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < 8; ++r) t += red[r][c];
    out[n] = t;
  }
}

static int colsum(const float* g, int64_t ld, int64_t M, int N, float* out, cudaStream_t s, bool deterministic = false) {
  if (deterministic) {
    colsum_det_kernel<<<(unsigned)((N + 31) / 32), 256, 0, s>>>(g, ld, M, N, out);
    CFN_LAUNCH_CHECK();
    return CFN_OK;
  }
  CFN_CUDA(cudaMemsetAsync(out, 0, (size_t)N * sizeof(float), s));
  const int rows = 256;
  colsum_kernel<<<(unsigned)((M + rows - 1) / rows), N < 256 ? ((N + 31) / 32) * 32 : 256, 0, s>>>(g, ld, M, N, out, rows);
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

// gradient range [lo, hi) that a single memset at the start of chain_network_bwd already zeroed (flat gradient buckets)
struct Zeroed {
  const float* lo = nullptr; const float* hi = nullptr;
  bool has(const float* q) const { return lo && q >= lo && q < hi; }
};

// K splits of the weight gradient dW(out_f x in_f) over M points, on the tensor cores (tc) or the CUDA cores; M < 0 gives
// the cap over every M (what the deterministic scratch is sized for)
static int64_t wgrad_split(bool tc, int64_t out_f, int64_t in_f, int64_t M) {
  int64_t split;
  if (tc) {
    // one K slice per CTA (pair): (m tiles x n tiles x splits) ~ number of SMs (pairs)
    const int cg = out_f <= 128 ? 1 : 2;
    const int64_t bn = in_f >= 256 ? 256 : ((in_f + 15) / 16) * 16;
    const int64_t tiles = ((out_f + 128 * cg - 1) / (128 * cg)) * ((in_f + bn - 1) / bn);
    split = (148 / cg) / tiles;
    if (M >= 0 && split > (M + 255) / 256) split = (M + 255) / 256;
  } else {
    const int64_t tiles = ((out_f + 127) / 128) * ((in_f + 127) / 128);
    split = (148 * 8 + tiles - 1) / tiles;
    if (M >= 0 && split > (M + 1023) / 1024) split = (M + 1023) / 1024;
  }
  return split < 2 ? 2 : split;             // split_k > 1 selects the atomic accumulate path
}

// floats of deterministic scratch (cfn_set_deterministic): the largest split x (out x in + out) over every weight gradient
// the backward chain issues, at the larger of the two engines' caps (a tensor-core handle falls back to the CUDA cores
// for a shape tgemm_supported rejects)
int64_t chain_det_scratch_floats(const CfnHandle* h) {
  int64_t need = 0;
  auto account = [&](int64_t out_f, int64_t in_f) {
    const int64_t split = std::max(wgrad_split(true, out_f, in_f, -1), wgrad_split(false, out_f, in_f, -1));
    need = std::max(need, split * (out_f * in_f + out_f));
  };
  for (size_t i = 0; i < h->slots.size(); ++i)
    if (h->wv[i].ld) account(h->slots[i].rows, h->wv[i].ld);
  account(3 * h->cfg.F, (h->cfg.h_alpha + 7) & ~7);    // amortisation matrices (padded K)
  account(15 * h->cfg.F, (h->cfg.h_rgb + 7) & ~7);
  return need;
}

// dW(out x in) = G(M x out)^T X(M x in), split over the point dimension, atomically accumulated into zeroed dW
// db (optional): the bias gradient = column sums of G, fused into the tensor-core GEMM when possible
static int wgrad(const CfnHandle* h, const float* G, int64_t ldg, int out_f, const float* X, int64_t ldx, int in_f, int64_t M,
                 float* dW, float* db, const Zeroed& zeroed, cudaStream_t s) {
  if (!h->deterministic && !zeroed.has(dW)) CFN_CUDA(cudaMemsetAsync(dW, 0, (size_t)out_f * in_f * sizeof(float), s));
  GemmArgs g{};
  g.A = G; g.a_rs = 1; g.a_cs = ldg;        // A(m=o, k=pt) = G[pt*ldg + o]
  g.B = X; g.b_rs = ldx; g.b_cs = 1;        // B(k=pt, n=i) = X[pt*ldx + i]
  g.C = dW; g.c_rs = in_f;
  g.M = out_f; g.N = in_f; g.K = M;
  g.ab_bf16 = h->chain_bf16; g.c_bf16 = 0;   // weight gradients are fp32
  g.split_k = 2;                             // (so that tgemm_supported sees the split-K flavour)
  g.split_k = (int)wgrad_split(h->gemm_tc && tgemm_supported(g), out_f, in_f, M);
  if (h->deterministic) { g.partials = h->det_scratch; g.partials_floats = h->det_floats; }
  if (db) {
    if (h->gemm_tc && tgemm_can_rowsum(g)) {
      if (!h->deterministic && !zeroed.has(db)) CFN_CUDA(cudaMemsetAsync(db, 0, (size_t)out_f * sizeof(float), s));
      g.rowsum = db;
    } else if (h->chain_bf16) {
      set_error("bf16 chain: the bias gradient could not be fused into the wgrad (out %d in %d)", out_f, in_f);
      return CFN_ESTATE;
    } else {
      int rc = colsum(G, ldg, M, out_f, db, s, h->deterministic != 0);
      if (rc) return rc;
    }
  }
  return gemm(h, g, 0, s);
}

// weight gradient of parameter slot `slot` (an nn.Linear whose input rows are X): straight into grads[slot] when the
// operand view is unpadded, otherwise through the padded scratch and two strided copies that drop the pad columns
static int wgrad_slot(const CfnHandle* h, int slot, const float* G, int64_t ldg, const float* X, int64_t ldx, int64_t M,
                      float* dW, float* db, float* scratch, const Zeroed& zeroed, cudaStream_t s) {
  const ParamSlot& w = h->slots[slot];
  const WView& v = h->wv[slot];
  if (v.ld == w.cols) return wgrad(h, G, ldg, w.rows, X, ldx, w.cols, M, dW, db, zeroed, s);
  int rc = wgrad(h, G, ldg, w.rows, X, ldx, v.ld, M, scratch, db, zeroed, s);
  if (rc) return rc;
  const int first = v.gap_at < w.cols ? v.gap_at : w.cols;
  if (first > 0)
    CFN_CUDA(cudaMemcpy2DAsync(dW, (size_t)w.cols * 4, scratch, (size_t)v.ld * 4, (size_t)first * 4, w.rows, cudaMemcpyDeviceToDevice, s));
  if (w.cols > first)
    CFN_CUDA(cudaMemcpy2DAsync(dW + first, (size_t)w.cols * 4, scratch + first + v.gap, (size_t)v.ld * 4,
                               (size_t)(w.cols - first) * 4, w.rows, cudaMemcpyDeviceToDevice, s));
  return CFN_OK;
}

// Gin(M x n_cols) = [accumulate +] Gout(M x out) W[:, col0:col0+n_cols], optional ReLU mask.  out_f32: Gin is fp32
// and is not rounded to the tf32 grid whatever the chain's storage (it is no later GEMM's operand: the input gradients)
static int dgrad(const CfnHandle* h, int slot, const float* Gout, int64_t ldgo, int col0, int n_cols, float* Gin,
                 int64_t ldgi, int64_t M, const float* mask, int64_t ld_mask, int accumulate, cudaStream_t s,
                 const uint32_t* mask_bits = nullptr, int bits_ld = 0, bool out_f32 = false) {
  const ParamSlot& w = h->slots[slot];
  const WView& v = h->wv[slot];
  GemmArgs g{};
  g.A = Gout; g.a_rs = ldgo; g.a_cs = 1;
  g.B = at(h, v.p, col0 + (col0 >= v.gap_at ? v.gap : 0)); g.b_rs = v.ld; g.b_cs = 1;   // B(k=o, n=i) = W[o*ld + col0' + i]
  g.C = Gin; g.c_rs = ldgi;
  g.aux = mask; g.aux_rs = ld_mask;
  g.aux_bits = mask ? mask_bits : nullptr; g.bits_ld = bits_ld;
  g.ab_bf16 = g.c_bf16 = h->chain_bf16;
  if (out_f32) g.c_bf16 = 0;
  g.M = M; g.N = n_cols; g.K = w.rows;
  g.epilogue = mask ? EPI_RELU_MASK_MUL : EPI_NONE;
  g.accumulate = accumulate; g.split_k = 1;
  return gemm(h, g, out_f32 ? 0 : 1, s);
}

// gradient tensors by parameter slot, passed BY VALUE as a kernel parameter: copying the table to the device from pageable
// host memory would make cudaMemcpyAsync synchronise the stream (and stall the host) once per training step
struct GradPtrs { float* p[64]; };

__global__ void scatter_rows_kernel(const float* __restrict__ dAm, const float* __restrict__ dAb, int cols,
                                    const int* __restrict__ gather, int rows, const GradPtrs grads) {
  int r = blockIdx.x;
  if (r >= rows) return;
  const int slot_w = gather[r * 4 + 0], slot_b = gather[r * 4 + 1], row = gather[r * 4 + 2];
  float* gw = grads.p[slot_w];
  float* gb = grads.p[slot_b];
  if (gw) for (int c = threadIdx.x; c < cols; c += blockDim.x) gw[(int64_t)row * cols + c] = dAm[r * cols + c];
  if (gb && threadIdx.x == 0) gb[row] = dAb[r];
}

int chain_input_grad_width(const CfnHandle* h) { return 2 * h->gp + h->gd; }

// grads == nullptr: no weight gradient at all (no wgrad, no scatter, no memset: a frozen network).  g_enc (M x
// chain_input_grad_width, fp32): when given, also the gradients of the encoded inputs, [g_gamma(p) through layer 0 |
// g_gamma(p) through the skip layer (zeros without one) | g_gamma(d) through the view layer], each block padded to gp /
// gp / gd columns (the pad columns meet zero weights and come out 0).
int chain_network_bwd(const CfnHandle* h, const float* g_flow_params, int64_t B, int N, float* ws, float* const* grads,
                      cudaStream_t s, float* g_enc) {
  const int64_t M = B * N;
  const int W = h->cfg.W, D = h->cfg.D, F = h->cfg.F, PP = h->PP;
  const int ha_n = h->cfg.h_alpha, hr_n = h->cfg.h_rgb;
  ChainLayout L = make_layout(h, M, 1);
  int rc;
  const bool want_w = grads != nullptr;
  const int ld_enc = chain_input_grad_width(h);
  if (want_w)
    for (int i = 4; i < (int)h->slots.size(); ++i)
      CFN_CHECK_ARG(grads[i] != nullptr, "cfn_network_bwd: grads[%d] (%s) is null", i, h->slots[i].name.c_str());
  float* dAm = ws + L.dAm;                       // (rows, cols) gathered weight grads
  float* dAb = dAm + (int64_t)PP * (ha_n > hr_n ? ha_n : hr_n);   // (rows) gathered bias grads

  // 1. through the tanh on the diagonals
  {
    int64_t total = M * PP;
    tanh_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(g_flow_params, ws + L.P, h->tanh_flags, ws + L.GP,
                                                                    total, PP, 3 * F, L.gpa, L.ldGP,
                                                                    h->chain_bf16 ? 2 : (h->gemm_tc ? 1 : 0));
    CFN_LAUNCH_CHECK();
  }
  const float* GPa = ws + L.GP;                   // gradient w.r.t. the alpha block of the (pre-tanh) flow record
  const float* GPc = at(h, ws + L.GP, L.gpa);     // ... and the rgb block
  const int ldGP = L.ldGP;
  LayerIO last = trunk_io(h, L, ws, M, D - 1, 1);
  const float* h7 = last.out;
  const int64_t ld7 = last.ld_out;
  float* G1 = ws + L.G1;
  float* G2 = ws + L.G2;
  float* gh = ws + L.gh;
  float* gv = ws + L.gv;
  float* dWp = ws + L.dWp;
  const bool bits = use_bits(h);
  // fused head dgrad: needs W_halpha stored right behind W_feat in the operand buffer with the same row stride
  const bool fuse_heads = h->wv[h->s_feat].ld == W && h->wv[h->s_halpha].ld == W &&
                          h->wv[h->s_halpha].p == at(h, h->wv[h->s_feat].p, (int64_t)W * W);
  const int64_t ld_g2 = fuse_heads ? W + ((ha_n + 7) & ~7) : W;
  float* gha = fuse_heads ? at(h, G2, W) : gh;                 // g_h_alpha lives in columns W.. of the g_feat rows when fused
  const int64_t ld_gha = fuse_heads ? ld_g2 : ha_n;
  const uint32_t* mbv = bits ? reinterpret_cast<const uint32_t*>(ws + L.mbv) : nullptr;
  auto MBl = [&](int layer) -> const uint32_t* {
    return bits ? reinterpret_cast<const uint32_t*>(ws + L.MB) + (int64_t)layer * M * L.bw : nullptr;
  };

  // Gradient tensors laid out back to back in slot order (cfnerf_b200.dist.FusedTrainStep's flat bucket): ONE memset
  // replaces the ~40 per-tensor ones of the split-K wgrads (each a graph node / launch of its own at 512 rays per step)
  Zeroed zeroed;
  if (want_w) {
    bool flat = true;
    for (size_t i = 5; i < h->slots.size(); ++i)
      flat = flat && (grads[i] == grads[4] + (h->slots[i].offset - h->slots[4].offset));
    if (flat) {
      const int64_t n = h->n_floats - h->slots[4].offset;
      CFN_CUDA(cudaMemsetAsync(grads[4], 0, (size_t)n * sizeof(float), s));
      zeroed.lo = grads[4];
      zeroed.hi = grads[4] + n;
    }
  }
  // zero every flow-conditioning gradient: rows the path never reads keep an exact 0 (SURVEY §0 fact 5)
  if (want_w && !zeroed.lo)
    for (int base : {h->s_frgb, h->s_falpha})
      for (int j = 0; j < 8; ++j)
        CFN_CUDA(cudaMemsetAsync(grads[base + j], 0, h->slots[base + j].numel * sizeof(float), s));

  // gradient pointers of every slot, handed to the scatter kernels by value
  GradPtrs table;
  for (size_t i = 0; i < 64; ++i) table.p[i] = (want_w && i < h->slots.size()) ? grads[i] : nullptr;

  // 2. alpha conditioning branch
  {
    // gathered dAmA = GP[:, :3F]^T ha ; bias = colsum
    if (want_w) {
      if ((rc = wgrad(h, GPa, ldGP, 3 * F, ws + L.ha, ha_n, ha_n, M, dAm, dAb, zeroed, s))) return rc;
      scatter_rows_kernel<<<3 * F, 64, 0, s>>>(dAm, dAb, ha_n, h->gatherA_dev, 3 * F, table);
      CFN_LAUNCH_CHECK();
    }
    // g_ha = GP[:, :3F] amA
    GemmArgs g{};
    g.A = GPa; g.a_rs = ldGP; g.a_cs = 1;
    g.B = h->amA_g; g.b_rs = ha_n; g.b_cs = 1;
    g.C = gha; g.c_rs = ld_gha; g.M = M; g.N = ha_n; g.K = 3 * F; g.split_k = 1;
    g.ab_bf16 = g.c_bf16 = h->chain_bf16;
    if ((rc = gemm(h, g, 1, s))) return rc;
    if (want_w && (rc = wgrad_slot(h, h->s_halpha, gha, ld_gha, h7, ld7, M, grads[h->s_halpha], grads[h->s_halpha + 1], dWp, zeroed, s))) return rc;
    // g_h7 (unmasked, first contribution) = g_ha W_halpha  -- or, fused, left for the K-concatenated GEMM of step 3
    if (!fuse_heads && (rc = dgrad(h, h->s_halpha, gha, ld_gha, 0, W, G1, W, M, nullptr, 0, 0, s))) return rc;
  }
  // 3. rgb conditioning branch
  {
    if (want_w) {
      if ((rc = wgrad(h, GPc, ldGP, 15 * F, ws + L.hr, hr_n, hr_n, M, dAm, dAb, zeroed, s))) return rc;
      scatter_rows_kernel<<<15 * F, 64, 0, s>>>(dAm, dAb, hr_n, h->gatherC_dev, 15 * F, table);
      CFN_LAUNCH_CHECK();
    }
    GemmArgs g{};
    g.A = GPc; g.a_rs = ldGP; g.a_cs = 1;
    g.B = h->amC_g; g.b_rs = hr_n; g.b_cs = 1;
    g.C = gh; g.c_rs = hr_n; g.M = M; g.N = hr_n; g.K = 15 * F; g.split_k = 1;
    g.ab_bf16 = g.c_bf16 = h->chain_bf16;
    if ((rc = gemm(h, g, 1, s))) return rc;
    if (want_w && (rc = wgrad_slot(h, h->s_hrgb, gh, hr_n, ws + L.v, W / 2, M, grads[h->s_hrgb], grads[h->s_hrgb + 1], dWp, zeroed, s))) return rc;
    // g_v = (g_hr W_hrgb) * relu'(v)
    if ((rc = dgrad(h, h->s_hrgb, gh, hr_n, 0, W / 2, gv, W / 2, M, ws + L.v, W / 2, 0, s, mbv, L.bwv))) return rc;
    if (want_w && (rc = wgrad_slot(h, h->s_views, gv, W / 2, ws + L.V, L.ldv, M, grads[h->s_views], grads[h->s_views + 1], dWp, zeroed, s))) return rc;
    // g_gamma(d) = g_v W_view[:, W:W+in_dir], only when the input gradients are asked for
    if (g_enc && (rc = dgrad(h, h->s_views, gv, W / 2, W, h->gd, g_enc + 2 * h->gp, ld_enc, M, nullptr, 0, 0, s, nullptr, 0, true))) return rc;
    // g_feat = g_v W_view[:, :W]
    if ((rc = dgrad(h, h->s_views, gv, W / 2, 0, W, G2, ld_g2, M, nullptr, 0, 0, s))) return rc;
    if (want_w && (rc = wgrad_slot(h, h->s_feat, G2, ld_g2, h7, ld7, M, grads[h->s_feat], grads[h->s_feat + 1], dWp, zeroed, s))) return rc;
    if (fuse_heads) {
      // g_h7 = ([g_feat | g_ha] [W_feat ; W_halpha]) * relu'(h7): one GEMM over the concatenated K instead of a second,
      // accumulating one (its read-modify-write of g_h7 cost three times a plain dgrad)
      GemmArgs g{};
      g.A = G2; g.a_rs = ld_g2; g.a_cs = 1;
      g.B = h->wv[h->s_feat].p; g.b_rs = W; g.b_cs = 1;       // rows 0..W-1 = W_feat, rows W.. = W_halpha (adjacent in wg)
      g.C = G1; g.c_rs = W;
      g.aux = h7; g.aux_rs = ld7; g.aux_bits = MBl(D - 1); g.bits_ld = L.bw;
      g.M = M; g.N = W; g.K = W + ha_n;
      g.epilogue = EPI_RELU_MASK_MUL; g.split_k = 1;
      g.ab_bf16 = g.c_bf16 = h->chain_bf16;
      if ((rc = gemm(h, g, 1, s))) return rc;
    } else {
      // g_h7 = (g_h7 + g_feat W_feat) * relu'(h7)
      if ((rc = dgrad(h, h->s_feat, G2, W, 0, W, G1, W, M, h7, ld7, 1, s, MBl(D - 1), L.bw))) return rc;
    }
  }
  // 4. trunk, last layer to first
  float* gout = G1;
  float* gin = G2;
  for (int i = D - 1; i >= 0; --i) {
    LayerIO io = trunk_io(h, L, ws, M, i, 1);
    const int slot = h->s_pts(i, 0);
    if (want_w && (rc = wgrad_slot(h, slot, gout, W, io.in, io.ld_in, M, grads[slot], grads[slot + 1], dWp, zeroed, s))) return rc;
    if (g_enc && (i == 0 || (h->skip >= 0 && i == h->skip + 1))) {
      // g_gamma(p) = dY_i W_i[:, 0:in_pos] (+ gap / pad columns, zero weights): layer 0, and the skip layer whose input is
      // cat[gamma(p), h]; separate column blocks (the bf16 chain has no accumulating GEMM), added by the ray kernel
      if ((rc = dgrad(h, slot, gout, W, 0, h->gp, g_enc + (i == 0 ? 0 : h->gp), ld_enc, M, nullptr, 0, 0, s, nullptr, 0, true))) return rc;
    }
    if (i == 0) break;
    // gradient w.r.t. the previous layer's (post-ReLU) output, masked by its ReLU
    LayerIO prev = trunk_io(h, L, ws, M, i - 1, 1);
    const int col0 = (h->skip >= 0 && i == h->skip + 1) ? h->in_pos : 0;   // skip input is cat[gamma(p), h]
    if ((rc = dgrad(h, slot, gout, W, col0, W, gin, W, M, prev.out, prev.ld_out, 0, s, MBl(i - 1), L.bw))) return rc;
    float* t = gout; gout = gin; gin = t;
  }
  if (g_enc && h->skip < 0)
    CFN_CUDA(cudaMemset2DAsync(g_enc + h->gp, (size_t)ld_enc * 4, 0, (size_t)h->gp * 4, (size_t)M, s));
  return CFN_OK;
}

}  // namespace cfn
