// K5-TC — general strided GEMM on the 5th-generation tensor cores, TMA-fed, fp32 accumulation in TMEM.
//
//   C(m,n) = epi( [C(m,n) +] sum_k A(m,k) B(k,n) + bias[n] )        (same contract as sgemm.cu's launch_sgemm)
//
// Two storage flavours of the operands (template parameter DT):
//   DT = 0  fp32 storage, tcgen05.mma kind::tf32 (K = 8 per instruction)   — CFN_PREC_TF32 and the tf32 training chain
//   DT = 1  bf16 storage, tcgen05.mma kind::f16  (K = 16 per instruction)  — the bf16 training chain (CFN_PREC_BF16)
// This is the contraction of the TRAINING path (forward with saved activations, dgrad chain, split-K wgrad;
// reference: loss.backward() through model/models.py:165-186, run_nerf_uncertainty_NF.py:1065-1067) and of the
// CFN_PREC_TF32 render mode.  Operands stay row-major in HBM exactly where mlp_chain.cu's orchestration keeps them,
// so the three GEMM flavours of a Linear need no transposed copies:
//   forward   Y = X W^T      A = X  (K-major)   B = W  (K-major)
//   dgrad     dX = dY W      A = dY (K-major)   B = W  (N-major: tcgen05 "MN-major" operand)
//   wgrad     dW = dY^T X    A = dY (M-major)   B = X  (N-major), K = points, split over CTAs, fp32 atomics
// Both majors are fed by the same kind of TMA tensor map over the row-major buffers (boxes with 128 contiguous bytes);
// only the shared-memory matrix descriptor and the instruction descriptor's major bits differ.  MN-major layouts:
// 32-bit operands need SWIZZLE_128B_BASE32B (TMA 128B_ATOM_32B), 16-bit operands the ordinary SWIZZLE_128B.
//
// Structure: persistent CTAs (or CTA pairs, cta_group::2: M = 256 rows per pair, each CTA stages half of B), tiles
// of 128 x bn (bn <= 256) accumulated in TMEM, TWO accumulator buffers (2 x 256 columns) so the epilogue of tile i
// overlaps the MMAs of tile i+1; a ring of TMA stages (A 16 KB + B <= 32 KB per 128-byte K block); warp roles:
// 4 * EPW epilogue warps (EPW = 2 for fp32 storage, 4 for bf16), TMEM allocator, TMA producer, MMA issuer.
// Out-of-range rows / columns / K tails are zero-filled by the TMA (the tensor maps carry the logical extents).
#include <cuda.h>
#include <cuda_bf16.h>

#include <math.h>

#include "common.cuh"
#include "ptx_sm100.cuh"

namespace cfn {
namespace {

// warps: 4 * EPW epilogue warps (EPW per TMEM lane quarter), then allocator, (spare), TMA producer, MMA issuer.
// fp32 storage: EPW = 2 (the MMAs of a tile take 8192 cycles, two warps per quarter drain it in time);
// bf16 storage: EPW = 4 (4096 cycles per tile: with two warps per quarter the epilogue, not the MMA, set the tile time)
__host__ __device__ constexpr int tg_epw(int dt) { return dt ? 4 : 2; }
__host__ __device__ constexpr int tg_threads(int dt) { return (4 * tg_epw(dt) + 4) * 32; }
constexpr int TG_MAX_STAGES = 6;
constexpr int TG_A_BYTES = 128 * 128;   // 128 rows x 32 floats
constexpr int TG_STG_LD = 36;           // floats per row of an epilogue staging tile (32 + 4: conflict-free float4 rows)
__host__ __device__ constexpr int tg_stg_bytes(int dt) { return 4 * tg_epw(dt) * 32 * TG_STG_LD * 4; }   // one 32 x 32 tile per epilogue warp

struct TgParams {
  float* C; int64_t c_rs;
  const float* bias; const float* aux; int64_t aux_rs;
  int64_t M; int N; int64_t K;
  int epilogue, accumulate, split_k, atomic, round_out, vec_ok;
  int vec8_ok;         // bf16 C: rows are 16-byte addressable in groups of 8 columns (the lean bf16 epilogue)
  int bn;              // N of one tcgen05.mma (multiple of 16, <= 256)
  int b_rows_cta;      // B rows (n) staged by one CTA = bn / CG
  int b_blocks;        // N-major B: 32-column blocks staged by one CTA
  int64_t k_per_split; // multiple of 32
  int64_t m_tiles; int n_tiles;
  int64_t n_work;      // m_tiles * n_tiles * split_k
  int stages; int stage_bytes;
  float* rowsum;       // optional (atomic GEMMs): rowsum[m] += sum_k A(m,k)
  int64_t partial_stride;   // split-K without atomics (deterministic mode): split z STORES its tile at C + z * partial_stride
                            // (and its row sums at rowsum + z * M); the caller adds the slabs in a fixed order afterwards
  uint32_t* mask_out;  // optional (EPI_RELU): word [m][n / 32], bit 8 * (n % 4) + (n % 32) / 4 = output (m, n) > 0
  const uint32_t* aux_bits;   // optional (EPI_RELU_MASK_MUL): the same words, read instead of the fp32 aux
  int64_t bits_ld;     // words per row of either
};

using namespace ptx;   // mbarrier / cluster / TMA / tcgen05 wrappers shared with mlp_tc.cu (ptx_sm100.cuh)

// DT = 0: fp32 storage, kind::tf32 (K = 8 per instruction); DT = 1: bf16 storage, kind::f16 (K = 16)
template <int CG, int DT>
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  if (CG == 1 && DT == 0)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
  else if (CG == 2 && DT == 0)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
  else if (CG == 1)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// round-to-nearest (ties away) onto the 10-bit tf32 significand: the tensor core TRUNCATES fp32 operands, which is
// a one-sided error that accumulates over the layers; operands written through this are read back exactly
__device__ __forceinline__ float round_tf32(float x) {
  uint32_t r; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x)); return __uint_as_float(r);
}

// two fp32 -> packed bf16 pair (lo = first column), optional fused ReLU
template <bool RELU>
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t d;
  if (RELU) asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  else asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}

struct TgBarriers {
  uint64_t full[TG_MAX_STAGES];
  uint64_t empty[TG_MAX_STAGES];
  uint64_t acc_full[2];
  uint64_t acc_empty[2];
  uint32_t tmem_ptr;
  uint32_t pad;
};

// descriptor constants (cute::UMMA::SmemDescriptor): version 1 (bit 46), SWIZZLE_128B (2 << 61)
//   K-major : rows of 128 bytes, 8-row groups 1024 bytes apart (SBO), LBO unused (1)
//   MN-major: for 32-bit operands the only layout is SWIZZLE_128B_BASE32B (layout type 1; TMA swizzle 128B_ATOM_32B: the
//             32-byte units of a 128-byte row are permuted by row % 4): 32-float column blocks `lbo` bytes apart (LBO),
//             4-k-row groups 512 bytes apart (SBO)   (cute::UMMA::Layout_MN_SW128_32B_Atom)
__device__ __forceinline__ uint64_t desc_hi_kmajor() {
  return ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
__device__ __forceinline__ uint64_t desc_hi_mnmajor(uint32_t lbo_bytes) {
  return ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(512 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)1 << 61);
}
// 16-bit operands, MN-major: the ordinary SWIZZLE_128B (type 2), 64-element column blocks `lbo` bytes apart, 8-k-row
// groups 1024 bytes apart (cute::UMMA::Layout_MN_SW128_Atom)
__device__ __forceinline__ uint64_t desc_hi_mnmajor16(uint32_t lbo_bytes) {
  return ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}

// EPI (compile-time epilogue flavour: one instruction stream per flavour keeps the epilogue loop short enough to unroll)
enum { TG_PLAIN = 0, TG_RELU = 1, TG_TANH = 2, TG_MASK = 3, TG_ATOMIC = 4 };

template <int CG, bool A_MN, bool B_MN, int EPI, int DT, bool CBF>
__global__ void __launch_bounds__(tg_threads(DT), 1)
tgemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TgParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = smem_u32(smem_raw);
  if (smem_base & 1023u) __trap();
  TgBarriers* bars = reinterpret_cast<TgBarriers*>(smem_raw + (size_t)p.stages * p.stage_bytes);

  constexpr int EPW = tg_epw(DT), TG_THREADS = tg_threads(DT);
  constexpr int TG_W_ALLOC = 4 * EPW, TG_W_TMA = 4 * EPW + 2, TG_W_MMA = 4 * EPW + 3;
  constexpr int BKE = DT ? 64 : 32;            // elements per 128-byte K block
  constexpr int MNB = DT ? 64 : 32;            // elements per 128-byte row of an MN-major block
  constexpr uint32_t MN_BLOCK_BYTES = BKE * 128;   // one MN-major block: BKE k rows of 128 bytes
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;
  const int64_t unit0 = blockIdx.x / CG, n_grid_units = gridDim.x / CG;
  auto bar_local = [&](const uint64_t* b) { return smem_u32(b); };
  auto bar_leader = [&](const uint64_t* b) { return (CG == 2) ? mapa_rank(smem_u32(b), 0) : smem_u32(b); };

  if (threadIdx.x == 0) {
    for (int s = 0; s < TG_MAX_STAGES; ++s) { mbar_init(bar_local(&bars->full[s]), CG); mbar_init(bar_local(&bars->empty[s]), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(bar_local(&bars->acc_full[b]), 1); mbar_init(bar_local(&bars->acc_empty[b]), 4 * EPW * CG); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // 2 KB of ones right after the barriers: the B operand of the optional row-sum MMA (any layout of ones is ones)
  const uint32_t ones_addr = smem_base + (uint32_t)p.stages * p.stage_bytes + 1024u;
  if (EPI == TG_ATOMIC && p.rowsum) {
    uint32_t* ones = reinterpret_cast<uint32_t*>(smem_raw + (size_t)p.stages * p.stage_bytes + 1024);
    for (int i = threadIdx.x; i < 512; i += TG_THREADS) ones[i] = DT ? 0x3F803F80u : 0x3F800000u;   // bf16 pairs / fp32
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == TG_W_ALLOC) {
    if (CG == 1) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&bars->tmem_ptr)), "r"(512) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&bars->tmem_ptr)), "r"(512) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars->tmem_ptr);

  // work item w -> (m tile, n tile, K split): n fastest, so the n tiles of one row panel run side by side (A from L2)
  auto decode = [&](int64_t w, int64_t& mt, int& nt, int& z) {
    nt = (int)(w % p.n_tiles);
    const int64_t r = w / p.n_tiles;
    mt = r % p.m_tiles;
    z = (int)(r / p.m_tiles);
  };
  auto k_blocks = [&](int z, int64_t& k_begin) {
    k_begin = (int64_t)z * p.k_per_split;
    int64_t k_end = k_begin + p.k_per_split;
    if (k_end > p.K) k_end = p.K;
    return (int)((k_end - k_begin + BKE - 1) / BKE);
  };

  if (warp == TG_W_TMA) {
    // ================================= TMA producer =================================
    int stage = 0; uint32_t phase = 0;
    const uint32_t b_tx = B_MN ? (uint32_t)p.b_blocks * MN_BLOCK_BYTES : (uint32_t)p.b_rows_cta * 128u;
    for (int64_t w = unit0; w < p.n_work; w += n_grid_units) {
      int64_t mt; int nt, z; decode(w, mt, nt, z);
      int64_t k_begin; const int nkb = k_blocks(z, k_begin);
      const int m0 = (int)(mt * 128 * CG + rank * 128);
      const int n0 = nt * p.bn + (int)rank * p.b_rows_cta;
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(bar_local(&bars->empty[stage]), phase ^ 1u);
        if (elect_one()) {
          const uint32_t full_bar = bar_local(&bars->full[stage]);
          if (rank == 0) mbar_expect_tx(full_bar, (uint32_t)(TG_A_BYTES + b_tx) * CG);
          else mbar_arrive_cluster(bar_leader(&bars->full[stage]));
          const uint32_t dstA = smem_base + (uint32_t)stage * p.stage_bytes;
          const uint32_t dstB = dstA + TG_A_BYTES;
          const int k0 = (int)(k_begin + (int64_t)kb * BKE);
          if (!A_MN) tma_load_2d<CG>(dstA, &tmA, k0, m0, full_bar);
          else {
#pragma unroll
            for (int j = 0; j < 128 / MNB; ++j) tma_load_2d<CG>(dstA + j * MN_BLOCK_BYTES, &tmA, m0 + MNB * j, k0, full_bar);
          }
          if (!B_MN) tma_load_2d<CG>(dstB, &tmB, k0, n0, full_bar);
          else
            for (int j = 0; j < p.b_blocks; ++j) tma_load_2d<CG>(dstB + j * MN_BLOCK_BYTES, &tmB, n0 + MNB * j, k0, full_bar);
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == TG_W_MMA) {
    // ================================= MMA issuer (leader CTA; whole warp walks, one elected lane issues) ============
    if (rank == 0) {
      int stage = 0; uint32_t phase = 0;
      // instruction descriptor (cute::UMMA::InstrDescriptor): D = f32 (1 << 4), A/B = tf32 (2), major bits 15 / 16
      constexpr uint32_t FMT = DT ? 1u : 2u;   // bf16 : tf32
      const uint32_t idesc = (1u << 4) | (FMT << 7) | (FMT << 10) | ((A_MN ? 1u : 0u) << 15) | ((B_MN ? 1u : 0u) << 16) |
                             ((uint32_t)(p.bn >> 3) << 17) | ((uint32_t)((128 * CG) >> 4) << 24);
      const uint64_t mn_hi = DT ? desc_hi_mnmajor16(MN_BLOCK_BYTES) : desc_hi_mnmajor(MN_BLOCK_BYTES);
      const uint64_t a_hi = A_MN ? mn_hi : desc_hi_kmajor();
      const uint64_t b_hi = B_MN ? mn_hi : desc_hi_kmajor();
      // one MMA K slice (8 tf32 / 16 bf16 elements): 32 bytes along a K-major row, or 8 / 16 k rows of an MN-major block
      constexpr uint32_t MN_STEP = (DT ? 2048u : 1024u) >> 4;
      const uint32_t a_step = A_MN ? MN_STEP : (32u >> 4);
      const uint32_t b_step = B_MN ? MN_STEP : (32u >> 4);
      const uint32_t idesc16 = (idesc & ~(0x3Fu << 17)) | ((16u >> 3) << 17);
      const uint64_t ones_desc = b_hi | (uint64_t)((ones_addr & 0x3FFFFu) >> 4);
      uint32_t it = 0;
      for (int64_t w = unit0; w < p.n_work; w += n_grid_units, ++it) {
        int64_t mt; int nt, z; decode(w, mt, nt, z);
        int64_t k_begin; const int nkb = k_blocks(z, k_begin);
        const uint32_t buf = it & 1u;
        mbar_wait(bar_local(&bars->acc_empty[buf]), ((it >> 1) & 1u) ^ 1u);   // the epilogue drained this buffer
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * 256u;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(bar_local(&bars->full[stage]), phase);
          tc_fence_after();
          const uint32_t a_addr = smem_base + (uint32_t)stage * p.stage_bytes;
          const uint32_t b_addr = a_addr + TG_A_BYTES;
          const uint64_t adesc = a_hi | (uint64_t)((a_addr & 0x3FFFFu) >> 4);
          const uint64_t bdesc = b_hi | (uint64_t)((b_addr & 0x3FFFFu) >> 4);
          if (elect_one()) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks)
              umma_tf32<CG, DT>(d_tmem, adesc + (uint64_t)(a_step * ks), bdesc + (uint64_t)(b_step * ks), idesc, (kb > 0 || ks > 0) ? 1u : 0u);
            if (EPI == TG_ATOMIC && p.rowsum && nt == 0) {   // columns 256.. are free: a row-sum GEMM owns one work item per CTA (pair)
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                umma_tf32<CG, DT>(tmem_base + 256u, adesc + (uint64_t)(a_step * ks), ones_desc, idesc16, (kb > 0 || ks > 0) ? 1u : 0u);
            }
            umma_commit<CG>(bar_local(&bars->empty[stage]));
          }
          __syncwarp();
          if (++stage == p.stages) { stage = 0; phase ^= 1u; }
        }
        if (elect_one()) umma_commit<CG>(bar_local(&bars->acc_full[buf]));
        __syncwarp();
      }
    }
  } else if (warp < 4 * EPW) {
    // ================================= epilogue warps =================================
    const int q = warp & 3, hh = warp >> 2;
    float* stg = reinterpret_cast<float*>(smem_raw + (size_t)p.stages * p.stage_bytes + 3072) + warp * (32 * TG_STG_LD);
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t it = 0;
    const int sub_r = lane >> 3, c4 = (lane & 7) * 4;
    for (int64_t w = unit0; w < p.n_work; w += n_grid_units, ++it) {
      int64_t mt; int nt, z; decode(w, mt, nt, z);
      const uint32_t buf = it & 1u;
      const int64_t tile_m0 = mt * 128 * CG + rank * 128;
      const int n_tile0 = nt * p.bn;
      int n_cols = p.N - n_tile0; if (n_cols > p.bn) n_cols = p.bn;
      const int n_chunks = (n_cols + 31) / 32;
      // dgrad needs relu'(h) per output element.  The fast form is the BIT mask the forward GEMM wrote (one 32-bit word
      // per row and 32-column chunk): lane j holds the word of row j of this warp's 32 rows, the words of the next two
      // chunks are requested before they are needed (the first two before the accumulator is even waited for), so no
      // HBM round trip is exposed.  The fp32 form (aux = the saved activations) is kept for callers without bit masks.
      // The loops below are deliberately NOT unrolled: with every epilogue flavour inlined, an unrolled body ran out of
      // the instruction cache (a quarter of all stall samples were instruction fetches) and became the critical path.
      const bool use_bits = (EPI == TG_MASK) && p.aux_bits != nullptr;
      uint32_t pb1 = 0, pb2 = 0;
      auto load_bits = [&](int c) -> uint32_t {
        const int64_t gmp = tile_m0 + q * 32 + lane;
        return (gmp < p.M) ? __ldg(p.aux_bits + gmp * p.bits_ld + ((n_tile0 + c * 32) >> 5)) : 0u;
      };
      if (use_bits) {
        if (hh < n_chunks) pb1 = load_bits(hh);
        if (hh + EPW < n_chunks) pb2 = load_bits(hh + EPW);
      }
      mbar_wait(bar_local(&bars->acc_full[buf]), (it >> 1) & 1u);
      tc_fence_after();
#pragma unroll 1
      for (int c = hh; c < n_chunks; c += EPW) {
        // phase 1: this warp's 32 x 32 accumulator block, TMEM -> registers (thread = row) -> padded shared-memory tile
        {
          uint32_t v[32];
          tmem_ld32(tmem_row + buf * 256u + (uint32_t)(c * 32), v);
          tmem_ld_wait();
#pragma unroll
          for (int u = 0; u < 8; ++u)
            *reinterpret_cast<float4*>(stg + lane * TG_STG_LD + 4 * u) =
                make_float4(__uint_as_float(v[4 * u]), __uint_as_float(v[4 * u + 1]), __uint_as_float(v[4 * u + 2]), __uint_as_float(v[4 * u + 3]));
        }
        __syncwarp();
        const uint32_t curb = pb1;
        if (use_bits) {
          pb1 = pb2;
          if (c + 2 * EPW < n_chunks) pb2 = load_bits(c + 2 * EPW);
        }
        // phase 2: 8 lanes per row, 4 rows per instruction: every global access of the warp is 4 full 128-byte lines
        const int gn = n_tile0 + c * 32 + c4;
        float b4[4] = {0.f, 0.f, 0.f, 0.f};
        uint32_t tanh_nib = 0;
        if (EPI != TG_ATOMIC) {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (gn + i < p.N) {
              if (p.bias) b4[i] = __ldg(p.bias + gn + i);
              if (EPI == TG_TANH && __ldg(p.aux + gn + i) != 0.f) tanh_nib |= 1u << i;
            }
        }
        const int64_t gm0 = tile_m0 + q * 32 + sub_r;
        // WARP-UNIFORM choice (both paths contain full-mask shuffles): the whole 32 x 32 block inside the matrix
        const bool block_inside = p.vec_ok && (tile_m0 + q * 32 + 31 < p.M) && (n_tile0 + c * 32 + 31 < p.N);
        if (CBF && (EPI == TG_PLAIN || EPI == TG_RELU || EPI == TG_MASK) && block_inside && p.vec8_ok && !p.accumulate) {
          // ---- bf16 output, lean form (the forward / dgrad GEMMs of the bf16 training chain): 4 lanes per row, 8 rows per
          // instruction, 8 columns = one 16-byte store per lane; bias + (ReLU fused into the conversion | mask select);
          // row pointers advance by a constant.  The general form below spent 11 instructions per element (ncu: issue
          // slots 61 % busy, the epilogue - not the MMAs or HBM - set the tile time); this one spends ~5.
          const int rr = lane >> 2, l4 = lane & 3, cg8 = l4 * 8;
          const int gn8 = n_tile0 + c * 32 + cg8;
          float bb[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) bb[i] = p.bias ? __ldg(p.bias + gn8 + i) : 0.f;
          const int64_t row0 = tile_m0 + q * 32 + rr;
          __nv_bfloat16* crow = reinterpret_cast<__nv_bfloat16*>(p.C) + row0 * p.c_rs + gn8;
          const int64_t cstep = 8 * p.c_rs;
          uint32_t* mrow = (EPI == TG_RELU && p.mask_out) ? p.mask_out + row0 * p.bits_ld + ((n_tile0 + c * 32) >> 5) : nullptr;
          const int64_t mstep = 8 * p.bits_ld;
          const int sh = 2 * l4;   // mask word: column n of the chunk is bit 8 * (n % 4) + n / 4; this lane owns n = cg8 .. cg8 + 7
          const float* srow = stg + rr * TG_STG_LD + cg8;
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float4 a0 = *reinterpret_cast<const float4*>(srow + t * 8 * TG_STG_LD);
            const float4 a1 = *reinterpret_cast<const float4*>(srow + t * 8 * TG_STG_LD + 4);
            float y[8] = {a0.x + bb[0], a0.y + bb[1], a0.z + bb[2], a0.w + bb[3], a1.x + bb[4], a1.y + bb[5], a1.z + bb[6], a1.w + bb[7]};
            if (EPI == TG_MASK && use_bits) {
              const uint32_t kw = __shfl_sync(0xffffffffu, curb, t * 8 + rr) >> sh;
#pragma unroll
              for (int i = 0; i < 8; ++i) y[i] = (kw & (1u << (8 * (i & 3) + (i >> 2)))) ? y[i] : 0.f;
            }
            uint4 pk;
            pk.x = pack_bf16x2<EPI == TG_RELU>(y[0], y[1]); pk.y = pack_bf16x2<EPI == TG_RELU>(y[2], y[3]);
            pk.z = pack_bf16x2<EPI == TG_RELU>(y[4], y[5]); pk.w = pack_bf16x2<EPI == TG_RELU>(y[6], y[7]);
            *reinterpret_cast<uint4*>(crow + t * cstep) = pk;
            if (EPI == TG_RELU && p.mask_out) {
              uint32_t m = 0;
#pragma unroll
              for (int i = 0; i < 8; ++i) m |= (y[i] > 0.f ? 1u : 0u) << (8 * (i & 3) + (i >> 2));
              m <<= sh;
              m |= __shfl_xor_sync(0xffffffffu, m, 1);
              m |= __shfl_xor_sync(0xffffffffu, m, 2);
              if (l4 == 0) mrow[t * mstep] = m;
            }
          }
        } else if (block_inside) {
          // ---- fast path: the whole 32 x 32 block is inside the matrix and 16-byte addressable ----
          const uint32_t sel_row = (uint32_t)sub_r | ((uint32_t)(4 + sub_r) << 4);   // byte sub_r of each vote pair
          uint32_t* mask_row = (EPI == TG_RELU && p.mask_out) ? p.mask_out + gm0 * p.bits_ld + ((n_tile0 + c * 32) >> 5) : nullptr;
#pragma unroll 4
          for (int t = 0; t < 8; ++t) {
            const int r = t * 4 + sub_r;
            const int64_t gm = gm0 + t * 4;
            const float4 a4 = *reinterpret_cast<const float4*>(stg + r * TG_STG_LD + c4);
            float x[4] = {a4.x, a4.y, a4.z, a4.w};
            float* cp = p.C + gm * p.c_rs + gn;
            if (EPI == TG_ATOMIC) {
              if (p.partial_stride) *reinterpret_cast<float4*>(cp + (int64_t)z * p.partial_stride) = make_float4(x[0], x[1], x[2], x[3]);
              else asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" :: "l"(cp), "f"(x[0]), "f"(x[1]), "f"(x[2]), "f"(x[3]) : "memory");
              continue;
            }
            uint32_t keep = 0x01010101u;   // relu'(h) of column slot i at bit 8 * i
            if (EPI == TG_MASK) {
              if (use_bits) keep = __shfl_sync(0xffffffffu, curb, r) >> (lane & 7);
              else if (p.epilogue == EPI_RELU_MASK_MUL) {
                const float4 t4 = __ldg(reinterpret_cast<const float4*>(p.aux + gm * p.aux_rs + gn));
                keep = (t4.x > 0.f ? 1u : 0u) | (t4.y > 0.f ? 0x100u : 0u) | (t4.z > 0.f ? 0x10000u : 0u) | (t4.w > 0.f ? 0x1000000u : 0u);
              }
              if (p.accumulate) { const float4 t4 = *reinterpret_cast<const float4*>(cp); x[0] += t4.x; x[1] += t4.y; x[2] += t4.z; x[3] += t4.w; }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              float y = x[i] + b4[i];
              if (EPI == TG_RELU) y = fmaxf(y, 0.f);
              if (EPI == TG_TANH) { if (tanh_nib & (1u << i)) y = tanhf(y); }
              if (EPI == TG_MASK) y = (keep & (1u << (8 * i))) ? y : 0.f;
              if (p.round_out) y = round_tf32(y);
              x[i] = y;
            }
            if (CBF) {
              // bf16 output: 4 columns = 8 bytes per lane, a row segment of 64 bytes per 8 lanes
              __nv_bfloat162 lo = __floats2bfloat162_rn(x[0], x[1]), hi = __floats2bfloat162_rn(x[2], x[3]);
              uint2 pk;
              pk.x = *reinterpret_cast<uint32_t*>(&lo); pk.y = *reinterpret_cast<uint32_t*>(&hi);
              *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.C) + gm * p.c_rs + gn) = pk;
            } else {
              *reinterpret_cast<float4*>(cp) = make_float4(x[0], x[1], x[2], x[3]);
            }
            if (EPI == TG_RELU && p.mask_out) {
              // relu'(y) of this row's 32 columns as one word: four warp votes (one per column slot) hold the bits of all
              // four rows of this instruction; three byte permutes pick this row's byte of each.  Layout (private to the
              // forward / dgrad pair): bit 8 * i + l of the word = column 4 * l + i of the 32-column chunk.
              const uint32_t v0 = __ballot_sync(0xffffffffu, x[0] > 0.f), v1 = __ballot_sync(0xffffffffu, x[1] > 0.f);
              const uint32_t v2 = __ballot_sync(0xffffffffu, x[2] > 0.f), v3 = __ballot_sync(0xffffffffu, x[3] > 0.f);
              const uint32_t word = __byte_perm(__byte_perm(v0, v1, sel_row), __byte_perm(v2, v3, sel_row), 0x5410);
              if ((lane & 7) == 0) mask_row[(int64_t)t * 4 * p.bits_ld] = word;
            }
          }
        } else {
          // ---- edge path: ragged rows / columns or unaligned C: element-wise, every lane still joins the shuffles ----
#pragma unroll 1
          for (int t = 0; t < 8; ++t) {
            const int r = t * 4 + sub_r;
            const int64_t gm = gm0 + t * 4;
            const float4 a4 = *reinterpret_cast<const float4*>(stg + r * TG_STG_LD + c4);
            const uint32_t rowbits = __shfl_sync(0xffffffffu, curb, r);
            const bool ok = gm < p.M && gn < p.N;
            float x[4] = {a4.x, a4.y, a4.z, a4.w};
            float* cp = p.C + gm * p.c_rs + gn;
            uint32_t pos = 0;
            if (ok) {
              uint32_t keep = 0x01010101u;
              if (EPI == TG_MASK) {
                if (use_bits) keep = rowbits >> (lane & 7);
                else if (p.epilogue == EPI_RELU_MASK_MUL) {
                  keep = 0;
#pragma unroll
                  for (int i = 0; i < 4; ++i) if (gn + i < p.N && __ldg(p.aux + gm * p.aux_rs + gn + i) > 0.f) keep |= 1u << (8 * i);
                }
              }
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                if (gn + i >= p.N) continue;
                if (EPI == TG_ATOMIC) {
                  if (p.partial_stride) cp[(int64_t)z * p.partial_stride + i] = x[i]; else atomicAdd(cp + i, x[i]);
                  continue;
                }
                float y = x[i] + b4[i];
                if (EPI == TG_MASK && p.accumulate) y += cp[i];
                if (EPI == TG_RELU) y = fmaxf(y, 0.f);
                if (EPI == TG_TANH) { if (tanh_nib & (1u << i)) y = tanhf(y); }
                if (EPI == TG_MASK) y = (keep & (1u << (8 * i))) ? y : 0.f;
                if (p.round_out) y = round_tf32(y);
                if (y > 0.f) pos |= 1u << (8 * i);
                if (CBF) reinterpret_cast<__nv_bfloat16*>(p.C)[gm * p.c_rs + gn + i] = __float2bfloat16_rn(y);
                else cp[i] = y;
              }
            }
            if (EPI == TG_RELU && p.mask_out) {
              uint32_t word = pos << (lane & 7);
              word |= __shfl_xor_sync(0xffffffffu, word, 1);
              word |= __shfl_xor_sync(0xffffffffu, word, 2);
              word |= __shfl_xor_sync(0xffffffffu, word, 4);
              if ((lane & 7) == 0 && gm < p.M) p.mask_out[gm * p.bits_ld + ((n_tile0 + c * 32) >> 5)] = word;
            }
          }
        }
        __syncwarp();   // the staging tile is rewritten by the next chunk
      }
      if (EPI == TG_ATOMIC && p.rowsum && nt == 0 && hh == 0) {
        const uint32_t sum = tmem_ld1(tmem_row + 256u);
        tmem_ld_wait();
        const int64_t gm = tile_m0 + q * 32 + lane;
        if (gm < p.M) {
          if (p.partial_stride) p.rowsum[(int64_t)z * p.M + gm] = __uint_as_float(sum);
          else atomicAdd(p.rowsum + gm, __uint_as_float(sum));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(bar_leader(&bars->acc_empty[buf]));
    }
  }

  // teardown: every MMA has completed (the epilogue waited for the last commit) and every TMA has been consumed
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == TG_W_ALLOC) {
    if (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(512) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(512) : "memory");
  }
}

// ---- host side -------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// row-major fp32 matrix (rows x cols, row stride ld floats) -> 2-D map with box {32 floats, box_rows}, SWIZZLE_128B
int make_map(CUtensorMap* map, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, bool mn_major, bool bf16) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    CFN_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    if (!p || q != cudaDriverEntryPointSuccess) { set_error("cuTensorMapEncodeTiled not available from the driver"); return CFN_ECUDA; }
    fn = (EncodeTiledFn)p;
  }
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * (bf16 ? 2 : 4)};
  cuuint32_t box[2] = {bf16 ? 64u : 32u, (cuuint32_t)box_rows};   // 128 bytes along the contiguous axis
  cuuint32_t estr[2] = {1, 1};
  // 32-bit MN-major operands need the 32-byte-atom flavour of the 128-byte swizzle; 16-bit ones the ordinary one
  CUresult r = fn(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, (mn_major && !bf16) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): rows %lld cols %lld ld %lld box_rows %d", (int)r, (long long)rows,
              (long long)cols, (long long)ld, box_rows);
    return CFN_ECUDA;
  }
  return CFN_OK;
}

bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

int num_sms() { return device_num_sms(); }   // per device (common.cuh)

template <int CG, bool A_MN, bool B_MN, int EPI, int DT = 0, bool CBF = false>
int launch_variant(const CUtensorMap& tmA, const CUtensorMap& tmB, const TgParams& p, size_t smem, cudaStream_t s) {
  // function attributes are PER DEVICE: one once-flag per device ordinal (a process may drive several GPUs)
  static PerDeviceOnce attr_set;
  auto kern = tgemm_kernel<CG, A_MN, B_MN, EPI, DT, CBF>;
  if (!attr_set.done()) {
    CFN_CUDA(cudaFuncSetAttribute((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set.mark();
  }
  int64_t units = num_sms() / CG;
  if (units > p.n_work) units = p.n_work;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(units * CG));
  cfg.blockDim = dim3(tg_threads(DT));
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, tmA, tmB, p);
  if (e != cudaSuccess) { set_error("tgemm_kernel launch failed: %s", cudaGetErrorString(e)); return CFN_ECUDA; }
  return CFN_OK;
}

}  // namespace

// Can this GEMM run on the TMA-fed tensor-core kernel?  (unit stride along one axis of each operand, 16-byte aligned
// bases and row strides; everything the network stage issues qualifies once its odd-width matrices are padded)
bool tgemm_supported(const GemmArgs& g) {
  if (g.M <= 0 || g.N <= 0 || g.K <= 0) return false;
  if (g.M > 0x7fffffff || g.K > 0x7fffffff) return false;
  const bool a_k = (g.a_cs == 1), a_mn = (g.a_rs == 1);
  const bool b_k = (g.b_rs == 1), b_mn = (g.b_cs == 1);
  if (!(a_k || a_mn) || !(b_k || b_mn)) return false;
  const int64_t a_ld = a_k ? g.a_rs : g.a_cs, b_ld = b_k ? g.b_cs : g.b_rs;
  const int epb = g.ab_bf16 ? 8 : 4;   // elements per 16 bytes
  if (a_ld % epb || b_ld % epb || a_ld <= 0 || b_ld <= 0) return false;
  if (!aligned16(g.A) || !aligned16(g.B)) return false;
  if (g.c_bf16 && !g.ab_bf16) return false;
  // instantiated (operand majors x epilogue) combinations: what the network stage issues
  const bool atomic = g.split_k > 1;
  const bool a_mn_ = !a_k, b_mn_ = !b_k;
  const bool plain = !atomic && g.epilogue == EPI_NONE && !g.accumulate;
  const bool mask = !atomic && (g.epilogue == EPI_RELU_MASK_MUL || (g.epilogue == EPI_NONE && g.accumulate));
  if (g.ab_bf16) {
    // bf16 storage: exactly the flavours of the training chain
    if (g.accumulate) return false;
    if (!a_mn_ && !b_mn_) return (plain && g.c_bf16) || (g.epilogue == EPI_RELU && g.c_bf16 && !atomic) || (g.epilogue == EPI_TANH_MASK && !g.c_bf16 && !atomic);
    if (!a_mn_ && b_mn_) return plain || (g.c_bf16 && mask && g.aux_bits != nullptr);   // fp32 C: the input dgrads
    if (a_mn_ && b_mn_) return atomic && !g.c_bf16;
    return false;
  }
  if (!a_mn_ && !b_mn_) return !atomic && (plain || mask || ((g.epilogue == EPI_RELU || g.epilogue == EPI_TANH_MASK) && !g.accumulate));
  if (!a_mn_ && b_mn_) return plain || mask;
  if (a_mn_ && b_mn_) return atomic || plain;
  return plain;
}

// tile / split / stage geometry of one GEMM
static void plan_tgemm(const GemmArgs& g, TgParams& p, int& CG, bool& a_mn, bool& b_mn, size_t& smem) {
  a_mn = (g.a_cs != 1);
  b_mn = (g.b_rs != 1);
  CG = (g.M <= 128) ? 1 : 2;
  p = TgParams{};
  p.C = g.C; p.c_rs = g.c_rs; p.bias = g.bias; p.aux = g.aux; p.aux_rs = g.aux_rs;
  p.M = g.M; p.N = g.N; p.K = g.K;
  p.epilogue = g.epilogue; p.accumulate = g.accumulate; p.split_k = g.split_k > 1 ? g.split_k : 1;
  const int bke = g.ab_bf16 ? 64 : 32;      // elements per 128-byte K block / MN-major row
  p.vec8_ok = g.c_bf16 && (g.c_rs % 8 == 0) && aligned16(g.C) && (g.epilogue != EPI_RELU_MASK_MUL || g.aux_bits != nullptr);
  if (g.c_bf16) p.vec_ok = (g.c_rs % 4 == 0) && (((uintptr_t)g.C & 7u) == 0);
  else p.vec_ok = (g.c_rs % 4 == 0) && aligned16(g.C) &&
                  (g.epilogue != EPI_RELU_MASK_MUL || g.aux_bits || (g.aux_rs % 4 == 0 && aligned16(g.aux)));
  int bn = (g.N + 15) / 16 * 16;
  if (bn > 256) bn = 256;
  p.bn = bn;
  p.b_rows_cta = bn / CG;
  p.b_blocks = (p.b_rows_cta + bke - 1) / bke;
  const int b_bytes = b_mn ? p.b_blocks * (bke * 128) : ((p.b_rows_cta * 128 + 1023) / 1024) * 1024;
  p.stage_bytes = TG_A_BYTES + b_bytes;
  const int stg_bytes = tg_stg_bytes(g.ab_bf16 ? 1 : 0);
  int stages = (int)((227 * 1024 - 3072 - stg_bytes) / p.stage_bytes);
  if (stages > TG_MAX_STAGES) stages = TG_MAX_STAGES;
  p.stages = stages;
  // split-K (wgrad): the caller pre-zeroes C and every split adds its partial sum with fp32 atomics
  p.atomic = g.split_k > 1 ? 1 : 0;
  int64_t kps = (g.K + p.split_k - 1) / p.split_k;
  kps = (kps + bke - 1) / bke * bke;
  p.k_per_split = kps;
  p.split_k = (int)((g.K + kps - 1) / kps);   // drop empty splits
  p.m_tiles = (g.M + 128 * CG - 1) / (128 * CG);
  p.n_tiles = (g.N + bn - 1) / bn;
  p.n_work = p.m_tiles * p.n_tiles * p.split_k;
  smem = (size_t)p.stages * p.stage_bytes + 3072 + stg_bytes;   // ring | barriers (1 KB) | ones (2 KB) | staging tiles
  if (smem < 120 * 1024) smem = 120 * 1024;   // one CTA per SM: each allocates all 512 TMEM columns
}

bool tgemm_can_rowsum(const GemmArgs& g) {
  if (!tgemm_supported(g) || g.split_k <= 1) return false;
  TgParams p; int CG; bool a_mn, b_mn; size_t smem;
  plan_tgemm(g, p, CG, a_mn, b_mn, smem);
  return p.n_work <= num_sms() / CG;
}

int launch_tgemm(const GemmArgs& g, int round_out, cudaStream_t s) {
  if (g.M == 0 || g.N == 0) return CFN_OK;
  CFN_CHECK_ARG(tgemm_supported(g), "tgemm: operand layout not supported by the TMA path");
  TgParams p; int CG; bool a_mn, b_mn; size_t smem;
  plan_tgemm(g, p, CG, a_mn, b_mn, smem);
  p.round_out = round_out;
  p.rowsum = g.rowsum;
  // deterministic split-K: the splits store dense (M x N) slabs into the caller's scratch, added in a fixed order below
  const bool det = p.atomic && g.partials != nullptr;
  float* const c_final = g.C;
  const int64_t c_rs_final = g.c_rs;
  float* const rowsum_final = g.rowsum;
  if (det) {
    const int64_t slab = g.M * (int64_t)g.N;
    CFN_CHECK_ARG((int64_t)p.split_k * (slab + (g.rowsum ? g.M : 0)) <= g.partials_floats,
                  "tgemm: deterministic split-K scratch too small (%lld floats needed)",
                  (long long)((int64_t)p.split_k * (slab + g.M)));
    p.C = g.partials; p.c_rs = g.N; p.partial_stride = slab;
    p.vec_ok = (g.N % 4 == 0) && aligned16(g.partials);
    if (g.rowsum) p.rowsum = g.partials + (int64_t)p.split_k * slab;
  }
  p.mask_out = (g.epilogue == EPI_RELU && !p.atomic) ? g.mask_out : nullptr;
  p.aux_bits = (g.epilogue == EPI_RELU_MASK_MUL) ? g.aux_bits : nullptr;
  p.bits_ld = g.bits_ld;
  CFN_CHECK_ARG(!g.rowsum || (p.atomic && p.n_work <= num_sms() / CG), "tgemm: rowsum needs one work item per CTA (see tgemm_can_rowsum)");

  CUtensorMap tmA, tmB;
  int rc;
  const bool bf = g.ab_bf16 != 0;
  const int bke = bf ? 64 : 32;
  if (!a_mn) rc = make_map(&tmA, g.A, g.M, g.K, g.a_rs, 128, false, bf);
  else rc = make_map(&tmA, g.A, g.K, g.M, g.a_cs, bke, true, bf);
  if (rc) return rc;
  if (!b_mn) rc = make_map(&tmB, g.B, g.N, g.K, g.b_cs, p.b_rows_cta, false, bf);
  else rc = make_map(&tmB, g.B, g.K, g.N, g.b_rs, bke, true, bf);
  if (rc) return rc;

  // epilogue flavour (compile-time in the kernel); only the combinations the network stage issues are instantiated,
  // anything else is reported as unsupported and the caller falls back to the CUDA-core engine
  int epi = TG_PLAIN;
  if (p.atomic) epi = TG_ATOMIC;
  else if (g.epilogue == EPI_RELU) epi = TG_RELU;
  else if (g.epilogue == EPI_TANH_MASK) epi = TG_TANH;
  else if (g.epilogue == EPI_RELU_MASK_MUL || g.accumulate) epi = TG_MASK;
  auto finish = [&](int rc_launch) -> int {
    if (rc_launch != CFN_OK || !det) return rc_launch;
    return reduce_split_partials(g.partials, p.split_k, g.M, g.N, c_final, c_rs_final,
                                 rowsum_final ? p.rowsum : nullptr, rowsum_final, s);
  };
#define TG_LAUNCH(cg, am, bm, e) return finish(launch_variant<cg, am, bm, e>(tmA, tmB, p, smem, s))
#define TG_BY_CG(am, bm, e) do { if (CG == 1) TG_LAUNCH(1, am, bm, e); else TG_LAUNCH(2, am, bm, e); } while (0)
#define TG_BF(am, bm, e, cbf) do { if (CG == 1) return finish(launch_variant<1, am, bm, e, 1, cbf>(tmA, tmB, p, smem, s)); \
                                   else return finish(launch_variant<2, am, bm, e, 1, cbf>(tmA, tmB, p, smem, s)); } while (0)
  if (bf) {
    if (!a_mn && !b_mn && epi == TG_PLAIN && g.c_bf16) TG_BF(false, false, TG_PLAIN, true);
    if (!a_mn && !b_mn && epi == TG_RELU && g.c_bf16) TG_BF(false, false, TG_RELU, true);
    if (!a_mn && !b_mn && epi == TG_TANH && !g.c_bf16) TG_BF(false, false, TG_TANH, false);
    if (!a_mn && b_mn && epi == TG_PLAIN && g.c_bf16) TG_BF(false, true, TG_PLAIN, true);
    if (!a_mn && b_mn && epi == TG_PLAIN && !g.c_bf16) TG_BF(false, true, TG_PLAIN, false);
    if (!a_mn && b_mn && epi == TG_MASK && g.c_bf16) TG_BF(false, true, TG_MASK, true);
    if (a_mn && b_mn && epi == TG_ATOMIC && !g.c_bf16) TG_BF(true, true, TG_ATOMIC, false);
  } else if (!a_mn && !b_mn) {
    if (epi == TG_PLAIN) TG_BY_CG(false, false, TG_PLAIN);
    if (epi == TG_RELU) TG_BY_CG(false, false, TG_RELU);
    if (epi == TG_TANH) TG_BY_CG(false, false, TG_TANH);
    if (epi == TG_MASK) TG_BY_CG(false, false, TG_MASK);
  } else if (!a_mn && b_mn) {
    if (epi == TG_PLAIN) TG_BY_CG(false, true, TG_PLAIN);
    if (epi == TG_MASK) TG_BY_CG(false, true, TG_MASK);
  } else if (a_mn && b_mn) {
    if (epi == TG_ATOMIC) TG_BY_CG(true, true, TG_ATOMIC);
    if (epi == TG_PLAIN) TG_BY_CG(true, true, TG_PLAIN);
  } else {
    if (epi == TG_PLAIN) TG_BY_CG(true, false, TG_PLAIN);
  }
#undef TG_BF
#undef TG_BY_CG
#undef TG_LAUNCH
  set_error("tgemm: operand-major / epilogue combination not instantiated (a_mn %d, b_mn %d, epilogue %d, split %d)",
            (int)a_mn, (int)b_mn, g.epilogue, g.split_k);
  return CFN_EINVAL;
}

}  // namespace cfn
