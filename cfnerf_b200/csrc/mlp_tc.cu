// K1 — the network stage on the 5th-generation tensor cores (CFN_PREC_BF16 / CFN_PREC_FP16).
//
// One persistent CTA pair per two SMs (cta_group::2, M = 256 points per pair, 128 TMEM lanes per CTA) walks tiles
// of 128 points per CTA through the WHOLE chain — positional encoding, 8x512 trunk with skip-concat, feature /
// view layers and the (pre-composed) conditioning heads — without the activations ever leaving the SM:
//   * gamma(p), gamma(d) are computed in registers and written straight into the swizzled shared-memory A tiles;
//   * every layer is a tcgen05.mma (kind::f16, fp32 accumulation in TMEM, N = 256 halves) over the 128x512 A tile
//     that stays resident in shared memory (128B-swizzled K-major chunks of 64 columns);
//   * the weights are ONE linear, pre-tiled bf16/fp16 stream in HBM/L2 that the TMA (cp.async.bulk.tensor,
//     SWIZZLE_128B) streams through a ring of shared-memory stages; with cta_group::2 each CTA loads half of every
//     weight tile, so the pair reads each weight byte once;
//   * the epilogue warps drain TMEM (tcgen05.ld), add the fp32 bias, apply ReLU, convert and store the next
//     layer's A chunk in place; per-chunk mbarriers let the next layer's MMAs start while the drain is running;
//   * the last two GEMMs emit the 18F conditional-flow parameters per point (tanh on the diagonals) to HBM.
// Because h_alpha_linear / h_rgb_linear feed the amortisation Linears with no nonlinearity in between
// (models.py:175,182 -> 366-368,380) they are composed into one matrix each at pack time (SURVEY §0 fact 3).
//
// Reference semantics: run_nerf_helpers.py:21-69 (embedding), model/models.py:165-186 (encode),
// model/models.py:358-385 (amortised parameters).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "handle.h"
#include "ptx_sm100.cuh"

namespace cfn {

// -DCFN_TC_ISSUE_STAMPS=1 (CFN_NVCC_EXTRA of cfnerf_b200/build.py): three clock64() stamps per ring slot in the MMA issuer
// instead of one — the diagnostic build behind scripts/r2_k1_issue.py; the stamps cost ~10 % of the kernel.
// -DCFN_TC_TIMELINE=1: the clock64() stamps behind scripts/k1_timeline.py (CFN_TC_PROFILE=1 at run time).
// Compiled OUT by default: predicated off they still cost 1.8 % of the kernel (same-box A/B, 17.36 -> 17.04 ms) - the
// single-warp producer / issuer loops are that sensitive to their instruction count.
#ifndef CFN_TC_TIMELINE
#define CFN_TC_TIMELINE 0
#endif
#ifndef CFN_TC_ISSUE_STAMPS
#define CFN_TC_ISSUE_STAMPS 0
#endif
constexpr int TC_MAX_STEPS = 20;
constexpr int TC_MAX_KCH = 12;
constexpr int TC_CHUNK_BYTES = 128 * 128;   // 128 rows x 64 columns x 2 bytes
constexpr int TC_SRC_GP = 8, TC_SRC_GD = 9;   // host-side source ids; the device sees ONE shared-memory chunk index AC:
                                              // gamma(p) and gamma(d) time-share one 16 KB tile (see TcPlanDev::gd_step)
constexpr int TC_THREADS = 384;             // warps 0..7 encode/epilogue, 8 TMEM alloc, 9 (profiling), 10 TMA, 11 MMA
constexpr int TC_W_ALLOC = 8, TC_W_WATCH = 9, TC_W_TMA = 10, TC_W_MMA = 11;   // the scheduler favours high warp ids
constexpr int TC_MAX_STAGES = 8;
constexpr int CG = 2;                       // cta_group::2: every tile of 256 points is shared by a CTA pair

struct TcStep {
  int kind;       // 0: bias+ReLU -> A tile, 1: bias -> A tile, 2: bias (+tanh where flagged) -> flow_params in HBM
  int n_total;    // padded output width (multiple of 16, <= 512)
  int n_part;     // N of one tcgen05.mma (<= 256)
  int n_parts;
  int order_rev;  // issue the parts in reverse order (lets a pending drain of TMEM columns 0..63 finish)
  int n_k;        // K chunks
  // per K chunk, packed: bits 0..15 offset of the A operand from the activation tile in 16-byte descriptor units
  // (chunk * 1024 + first K=16 slice * 2); bits 16..19 number of K=16 instructions; bits 20..23 shared-memory chunk
  // index (0..AC-1 activation chunk, AC = the gamma tile); bit 24: bias entry (its B tile is a [rows][16] SWIZZLE_32B
  // tile instead of a [rows][64] SWIZZLE_128B block); bit 25: the chunk reads gamma(d), which the epilogue warps write
  // into the gamma tile after step gd_step (wait for gd_ready); bits 26..29: split-commit steps, second part: after this
  // K chunk input chunk x (bit 26+x) has been read for the last time and may be overwritten by output chunk x
  unsigned int kinfo[TC_MAX_KCH];
  int bias_off;   // kind 2 only: floats into the table: bias[n_total] then tanh flags[n_total]
  int out_col;    // kind 2: first column in the flow-parameter record
  int n_valid;    // kind 2: valid output columns
  int row0;       // first row of this step's blocks in the weight stream (rows of 64 elements)
  // Two-part steps whose output overwrites the activation tile in place (kind 0/1, n_parts == 2, natural part order): the
  // accumulator of the FIRST part (columns 0..n_part-1 = output chunks 0..n_part/64-1) is committed on its own and
  // drained while the second part's MMAs run.  Output chunk x may only be stored once the second part has read INPUT
  // chunk x (kinfo bits 26..29).
  int split_commit;
};

struct TcPlanDev {
  int n_steps;
  int act_chunks;
  int stage_out;   // 1: the last step's outputs are staged in shared memory and written to HBM coalesced
  // ONE gamma tile: columns 0..62 hold gamma(p) and column 63 the constant 1 that multiplies every layer's bias row.
  // gamma(p) is dead once step gd_step (the skip layer, or layer 0 without a skip) has been accumulated: its epilogue
  // overwrites columns 0..31 with gamma(d) for the view layer.  The 16 KB this saves is a fifth weight stage.
  int gd_step;
  TcStep steps[TC_MAX_STEPS];
};

struct TcArgs {
  const float* rays; const float* z_vals; const float* pts; const float* viewdirs;
  int64_t M; int N; int L_pos; int L_dir;
  const float* table;   // biases / tanh flags
  float* flow_params; int PP;
  int64_t n_units;      // tiles of 128*CG points
  int stages; int stage_bytes;
  int stagger;                // cycles of start-up delay per CTA pair index (de-synchronises the weight-stream reads)
  unsigned long long* prof;   // optional timestamp buffer (CFN_TC_PROFILE=1): 4 roles x 4096 stamps of CTA 0
};

struct TcPlan {
  TcPlanDev dev;
  void* stream_dev;             // packed weight stream (2-byte elements)
  int64_t stream_rows;
  float* table_dev;             // biases + flags
  float* compA; float* compA_b; // composed alpha conditioning (3F x W), (3F)
  float* compC; float* compC_b; // composed rgb conditioning (15F x W/2), (15F)
  CUtensorMap tm_big, tm_small, tm_bias;
  int stages, stage_bytes, stagger;
  size_t smem_bytes;
  int num_sms;
  // pack recipe: one entry per 64-column block of the stream
  struct Block { int src; int row0, rows_valid, col0, cols_valid, rows_padded; int64_t stream_row; int bias_src; int bias_col; };
  std::vector<Block> blocks;
  int* blocks_dev;
  // bias recipe
  struct BiasSeg { int src; int n_valid; int n_padded; int off; int with_flags; int flag_off; };
  std::vector<BiasSeg> bias_segs;
  int table_floats;
  unsigned long long* prof_dev;
};

// ======================================================================================================
// PTX wrappers
// ======================================================================================================
using namespace ptx;   // mbarrier / cluster / TMA / tcgen05 wrappers shared with gemm_tc.cu (ptx_sm100.cuh)

__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
               :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}

// The four K=16 instructions of one 64-column K chunk in ONE asm block: the descriptors differ only in the start
// address field (+2 per 32 bytes of K), so the block takes the two low words and builds everything else itself.
__device__ __forceinline__ void umma_k64(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p, t;\n\t.reg .b64 da, db;\n\t.reg .b32 xa, xb;\n\t"
               "setp.ne.b32 p, %5, 0;\n\tsetp.eq.b32 t, %5, %5;\n\t"
               "mov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
               "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, p;\n\t"
               "add.u32 xa, %1, 2;\n\tadd.u32 xb, %2, 2;\n\tmov.b64 da, {xa, %3};\n\tmov.b64 db, {xb, %3};\n\t"
               "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, t;\n\t"
               "add.u32 xa, %1, 4;\n\tadd.u32 xb, %2, 4;\n\tmov.b64 da, {xa, %3};\n\tmov.b64 db, {xb, %3};\n\t"
               "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, t;\n\t"
               "add.u32 xa, %1, 6;\n\tadd.u32 xb, %2, 6;\n\tmov.b64 da, {xa, %3};\n\tmov.b64 db, {xb, %3};\n\t"
               "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, t;\n\t}"
               :: "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate) : "memory");
}

// two fp32 -> packed 16-bit pair (lo = element c, hi = element c+1), optional fused ReLU
template <bool FP16, bool RELU>
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  uint32_t d;
  if (FP16) {
    // .satfinite: an activation beyond the fp16 range (65504) saturates instead of becoming inf -> NaN downstream
    if (RELU) asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    else asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  } else {
    if (RELU) asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    else asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  }
  return d;
}

// shared-memory matrix descriptor: K-major, SWIZZLE_128B, 8-row groups 1024 bytes apart (cute::UMMA::SmemDescriptor)
__device__ __forceinline__ uint64_t make_sdesc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): fp32 accumulate, A/B = bf16 (1) or fp16 (0), both K-major
__device__ __forceinline__ uint32_t make_idesc(bool fp16, int M, int N) {
  const uint32_t fmt = fp16 ? 0u : 1u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// tanh through one exp and one fast division (abs error ~1e-6, far inside the operand rounding of this mode); the
// accurate tanhf costs ~40 dependent instructions per call and sat on the tile-boundary critical path
__device__ __forceinline__ float tanh_fast(float x) {
  const float t = __expf(2.0f * x);
  return 1.0f - __fdividef(2.0f, t + 1.0f);
}

// byte offset of the 16-byte unit u (0..7) of row r inside a 128B-swizzled 128x64 chunk
__device__ __forceinline__ uint32_t swz(int r, int u) { return (uint32_t)(r * 128 + ((u ^ (r & 7)) << 4)); }

constexpr int TC_PROF_N = 4096;
struct Prof {
  unsigned long long* p; int n;
  __device__ __forceinline__ void stamp() {
#if CFN_TC_TIMELINE
    if (p && n < TC_PROF_N) p[n++] = clock64();
#endif
  }
};

// ======================================================================================================
// the kernel
// ======================================================================================================
struct alignas(16) TcBarriers {   // the fp32 bias staging area follows it and is read as float4
  uint64_t full[TC_MAX_STAGES];
  uint64_t empty[TC_MAX_STAGES];
  uint64_t act_ready[8];
  uint64_t a_free[4];
  uint64_t acc_full;    // the step's accumulator (or its FIRST part in split-commit steps) is complete
  uint64_t acc_full2;   // split-commit steps: the second part is complete (its own barrier: the two commits of a short
                        // layer can be a few hundred cycles apart, and a waiter must never miss a phase)
  uint64_t out_done;
  uint64_t in_ready;
  uint64_t gd_ready;    // gamma(d) of the current tile has been written into the gamma tile
  uint32_t tmem_ptr;
  uint32_t pad;
};

// GD == false: gamma(p) of one row -> columns 0..62 of the gamma tile, column 63 = 1 (the bias column).
// GD == true : gamma(d) of one row -> columns 0..31 (27 values, zero padded); the other columns are left alone.
template <bool FP16, bool GD>
__device__ __forceinline__ void encode_row(float x, float y, float z, int L, uint32_t chunk_base, int r) {
  // [x, sin(2^l x), cos(2^l x)]_l in blocks of 3 (run_nerf_helpers.py:29-51), zero padded
  constexpr int NC = GD ? 32 : 64;
  constexpr int NL = GD ? 4 : 10;
  float e[NC];
#pragma unroll
  for (int i = 0; i < NC; ++i) e[i] = 0.f;
  e[0] = x; e[1] = y; e[2] = z;
  if (!GD) e[63] = 1.0f;   // multiplies the bias row of the weight stream
  // sin/cos of 2^l x by the double-angle recurrence from one accurate sincosf per coordinate: the absolute error
  // grows to ~2^9 * 1e-7 = 5e-5 at the top octave, far below the operand rounding of this mode (bf16 2e-3, fp16 5e-4)
  float sx, cx, sy, cy, sz, cz;
  sincosf(x, &sx, &cx); sincosf(y, &sy, &cy); sincosf(z, &sz, &cz);
#pragma unroll
  for (int l = 0; l < NL; ++l) {
    if (l < L) {
      e[3 + 6 * l + 0] = sx; e[3 + 6 * l + 1] = sy; e[3 + 6 * l + 2] = sz;
      e[3 + 6 * l + 3] = cx; e[3 + 6 * l + 4] = cy; e[3 + 6 * l + 5] = cz;
      float t;
      t = 2.0f * sx * cx; cx = fmaf(-2.0f * sx, sx, 1.0f); sx = t;
      t = 2.0f * sy * cy; cy = fmaf(-2.0f * sy, sy, 1.0f); sy = t;
      t = 2.0f * sz * cz; cz = fmaf(-2.0f * sz, sz, 1.0f); sz = t;
    }
  }
#pragma unroll
  for (int u = 0; u < NC / 8; ++u) {
    uint32_t p0 = pack2<FP16, false>(e[8 * u + 0], e[8 * u + 1]);
    uint32_t p1 = pack2<FP16, false>(e[8 * u + 2], e[8 * u + 3]);
    uint32_t p2 = pack2<FP16, false>(e[8 * u + 4], e[8 * u + 5]);
    uint32_t p3 = pack2<FP16, false>(e[8 * u + 6], e[8 * u + 7]);
    asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" :: "r"(chunk_base + swz(r, u)), "r"(p0), "r"(p1), "r"(p2), "r"(p3) : "memory");
  }
}

template <bool FP16>
__global__ void __launch_bounds__(TC_THREADS, 1)
mlp_tc_kernel(const __grid_constant__ CUtensorMap tm_big, const __grid_constant__ CUtensorMap tm_small,
              const __grid_constant__ CUtensorMap tm_bias,
              const __grid_constant__ TcPlanDev plan, const TcArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-byte alignment is required by SWIZZLE_128B; the dynamic segment is the only shared allocation
  const uint32_t smem_base = smem_u32(smem_raw);
  if (smem_base & 1023u) __trap();   // the dynamic segment is the only shared allocation: its base is 1024-aligned
  uint8_t* smem_gen = smem_raw;
  const int act_chunks = plan.act_chunks;
  const uint32_t act_base = smem_base;
  const uint32_t gp_base = act_base + act_chunks * TC_CHUNK_BYTES;
  const uint32_t stage_base = gp_base + TC_CHUNK_BYTES;
  TcBarriers* bars = reinterpret_cast<TcBarriers*>(smem_gen + (stage_base - smem_base) + (size_t)a.stages * a.stage_bytes);

  // the shuffle tells the compiler that `warp` is warp-uniform: the role branches below are then uniform branches and
  // the schedule arithmetic of the producer / issuer warps lives in the uniform datapath (no R2UR in front of every MMA)
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int64_t unit0 = blockIdx.x / CG, n_grid_units = gridDim.x / CG;

  // barrier addresses: local (shared::cta) and as seen on the pair's leader (shared::cluster)
  auto bar_local = [&](const uint64_t* b) { return smem_u32(b); };
  auto bar_leader = [&](const uint64_t* b) { return mapa_rank(smem_u32(b), 0); };

  if (threadIdx.x == 0) {
    for (int s = 0; s < TC_MAX_STAGES; ++s) { mbar_init(bar_local(&bars->full[s]), CG); mbar_init(bar_local(&bars->empty[s]), 1); }
    for (int j = 0; j < 8; ++j) mbar_init(bar_local(&bars->act_ready[j]), 4 * CG);
    for (int j = 0; j < 4; ++j) mbar_init(bar_local(&bars->a_free[j]), 1);
    mbar_init(bar_local(&bars->acc_full), 1);
    mbar_init(bar_local(&bars->acc_full2), 1);
    mbar_init(bar_local(&bars->out_done), 8 * CG);
    mbar_init(bar_local(&bars->in_ready), 4 * CG);
    mbar_init(bar_local(&bars->gd_ready), 4 * CG);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == TC_W_ALLOC) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(&bars->tmem_ptr)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(&bars->tmem_ptr);
  // All CTA pairs walk the SAME weight stream; started together they hit the same L2 lines at the same instant.
  // A one-off start-up skew (persistent kernel, uniform tiles: the skew persists) spreads the reads over the stream.
  // CFN_TC_STAGGER sets it and nothing else does, yet the prologue stays: without it the warp-role dispatch below is
  // compiled differently and K1 ran 0.6 % slower (fp16 17.29-17.32 -> 17.40-17.50 ms per 4.19 M points, same box;
  // B200 at 1000 W).
  if (a.stagger > 0) {
    const long long t0 = clock64();
    const long long wait = (long long)unit0 * a.stagger;
    while (clock64() - t0 < wait) { }
  }

  if (warp == TC_W_TMA) {
    // ================================= TMA producer (whole warp walks the schedule, one elected lane issues) ==========
    int stage = 0; uint32_t phase = 0;
    Prof prof{(a.prof && blockIdx.x == 0 && lane == 0) ? a.prof + 2 * TC_PROF_N : nullptr, 0};
    for (int64_t unit = unit0; unit < a.n_units; unit += n_grid_units) {
      for (int g = 0; g < plan.n_steps; ++g) {
        const TcStep& st = plan.steps[g];
        const int rows = st.n_part / CG;           // rows of each weight block this CTA stages
        const int n_blk = st.n_parts * st.n_k;
        for (int blk = 0; blk < n_blk; ++blk) {
          // (sleeping wait: polling this barrier with short probes instead cost 6 % of the kernel, round-2 A/B)
          mbar_wait(bar_local(&bars->empty[stage]), phase ^ 1u);
          prof.stamp();
          const bool bias_tile = (st.kinfo[blk % st.n_k] >> 24) & 1u;
          if (elect_one()) {
            const uint32_t full_bar = bar_local(&bars->full[stage]);   // peer bit cleared inside tma_load_2d
            const int row_g = st.row0 + blk * st.n_part + (int)rank * rows;
            const uint32_t dst = stage_base + (uint32_t)stage * a.stage_bytes;
            if (bias_tile) {
              // one K=16 slice: [rows][16] elements = 32 bytes per row, whole 128-row boxes (the tail of a short block
              // just re-reads the next rows of the stream; the MMA never touches them)
              const int n_box = (rows + 127) / 128;
              if (rank == 0) mbar_expect_tx(full_bar, (uint32_t)(n_box * 128 * 32 * CG));
              else mbar_arrive_cluster(bar_leader(&bars->full[stage]));
              for (int bx = 0; bx < n_box; ++bx) tma_load_2d<CG>(dst + bx * 128 * 32, &tm_bias, 0, row_g + bx * 128, full_bar);
            } else {
              if (rank == 0) mbar_expect_tx(full_bar, (uint32_t)(rows * 128 * CG));
              else mbar_arrive_cluster(bar_leader(&bars->full[stage]));
              int r = 0;
              for (; rows - r >= 128; r += 128) tma_load_2d<CG>(dst + r * 128, &tm_big, 0, row_g + r, full_bar);
              for (; r < rows; r += 16) tma_load_2d<CG>(dst + r * 128, &tm_small, 0, row_g + r, full_bar);
            }
          }
          __syncwarp();
          if (++stage == a.stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == TC_W_MMA) {
    // ================================= MMA issuer (leader CTA) =================================
    // The WHOLE warp runs the schedule so that every descriptor is a warp-uniform value; one elected lane issues.
    // Round-2 finding (profiles/README.md, "issuer timeline"): the loop below, not the tensor pipe or the weight ring,
    // set the pace of the kernel - ~575 cycles of dependent scalar code per ring slot whatever the slot's N.  The hot
    // path is therefore kept to: one table word per slot (host-packed descriptor offset / flags), one barrier test,
    // one fence, ONE asm block that issues the slot's four MMAs, one commit.
    if (rank == 0) {
      int stage = 0; uint32_t phase = 0;
      uint32_t act_gen = 0, in_cnt = 0, out_cnt = 0;
      bool pending_out = false, gd_seen = false;
      Prof prof{(a.prof && blockIdx.x == 0 && lane == 0) ? a.prof + 1 * TC_PROF_N : nullptr, 0};
      // Activation chunks of the current generation become ready in index order (0,1,2,...), and every generation is
      // consumed completely before the next one is produced, so one counter replaces per-chunk bookkeeping:
      // chunks [0, ready_upto) of generation act_gen are known to be written (and their TMEM columns drained).
      int ready_upto = 0;
      const uint32_t act_bar0 = bar_local(&bars->act_ready[0]);
      // short blocking probe first (wakes within tens of cycles), the sleeping wait only if that window passes
      auto wait_bar = [&](uint32_t bar, uint32_t parity) { if (!mbar_probe(bar, parity)) mbar_wait(bar, parity); };
      auto wait_act = [&](int j) {
        if (act_gen == 0) return;
        while (ready_upto <= j) {
          wait_bar(act_bar0 + 8u * ready_upto, (act_gen - 1u) & 1u);
          ++ready_upto;
        }
      };
      const uint32_t full_bar0 = bar_local(&bars->full[0]), empty_bar0 = bar_local(&bars->empty[0]);
      const uint32_t afree_bar0 = bar_local(&bars->a_free[0]);
      const uint32_t hi128 = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);   // SBO 1024 B, version 1, SWIZZLE_128B
      const uint32_t hi32 = (uint32_t)(256 >> 4) | (1u << 14) | (6u << 29);     // SBO 256 B, version 1, SWIZZLE_32B
      const uint32_t a_lo0 = ((act_base & 0x3FFFFu) >> 4) | (1u << 16);           // + LBO field (ignored for swizzled K-major)
      const uint32_t b_lo0 = ((stage_base & 0x3FFFFu) >> 4) | (1u << 16);
      const uint32_t b_step = (uint32_t)a.stage_bytes >> 4;
      const int n_stages = a.stages;      // a register copy: the asm memory clobbers made every use a fresh constant load
      uint32_t b_lo = b_lo0;
      bool cur_full = false;            // the full barrier of `stage` is already known complete
      for (int64_t unit = unit0; unit < a.n_units; unit += n_grid_units) {
        wait_bar(bar_local(&bars->in_ready), in_cnt & 1u); ++in_cnt;
        gd_seen = false;
        for (int g = 0; g < plan.n_steps; ++g) {
          const TcStep& st = plan.steps[g];
          const uint32_t idesc = make_idesc(FP16, 128 * CG, st.n_part);
          const int n_k = st.n_k, n_parts = st.n_parts;
          const bool split = st.split_commit != 0;
          for (int pi = 0; pi < n_parts; ++pi) {
            const int pp = st.order_rev ? (n_parts - 1 - pi) : pi;
            const int c0 = pp * st.n_part;
            if (pending_out && c0 < 64) { wait_bar(bar_local(&bars->out_done), (out_cnt - 1u) & 1u); pending_out = false; }
            {   // TMEM write-after-read: the columns of this part must have been drained
              int jl = (c0 + st.n_part - 1) / 64;
              if (jl > act_chunks - 1) jl = act_chunks - 1;
              wait_act(jl);
            }
            const uint32_t d_tmem = tmem_base + (uint32_t)c0;
            const bool commit_afree = split && pi == 1;
            // (Issuing several slots per elect block was tried: grouping everything ran 3 % slower - MMAs issued ahead of
            // the tensor pipe only take shared-memory bandwidth from the drain the next slots wait for - and grouping just
            // the small bias / head slots behind a leader was slower still.  One slot per iteration it is.)
            for (int kc = 0; kc < n_k; ++kc) {
              const uint32_t info = st.kinfo[kc];
              const int src = (info >> 20) & 0xf;
#if CFN_TC_ISSUE_STAMPS
              prof.stamp();      // diagnostic build: loop top (scripts/r2_k1_issue.py)
#endif
              if (src < act_chunks) { if (ready_upto <= src) wait_act(src); }
              else if (((info >> 25) & 1u) && !gd_seen) {   // gamma(d): written several layers ago, returns at once
                wait_bar(bar_local(&bars->gd_ready), (in_cnt - 1u) & 1u);
                gd_seen = true;
              }
              if (!cur_full) wait_bar(full_bar0 + 8u * stage, phase);
              prof.stamp();
              tc_fence_after();
              const uint32_t a_lo = a_lo0 + (info & 0xffffu);
              // the NEXT slot's weights: probed now, so that the barrier round trip overlaps the issue of this slot
              const int nstage = (stage + 1 == n_stages) ? 0 : stage + 1;
              const uint32_t nphase = (stage + 1 == n_stages) ? (phase ^ 1u) : phase;
              // (after the very last block this probes a phase that never completes: the short probe just returns false)
              const bool next_full = mbar_probe(full_bar0 + 8u * nstage, nphase);
              if (elect_one()) {
                const uint32_t nks = (info >> 16) & 0xfu;
                const uint32_t acc = kc > 0 ? 1u : 0u;
                if (nks == 4u) umma_k64(d_tmem, a_lo, b_lo, hi128, idesc, acc);
                else if ((info >> 24) & 1u)   // bias tile: K-major SWIZZLE_32B [rows][16], a single K=16 slice
                  umma(d_tmem, ((uint64_t)hi128 << 32) | a_lo, ((uint64_t)hi32 << 32) | b_lo, idesc, acc);
                else
                  for (uint32_t ks = 0; ks < nks; ++ks)
                    umma(d_tmem, ((uint64_t)hi128 << 32) | (a_lo + 2u * ks), ((uint64_t)hi128 << 32) | (b_lo + 2u * ks), idesc,
                         (acc || ks > 0) ? 1u : 0u);
                umma_commit<CG>(empty_bar0 + 8u * stage);
                if (commit_afree) {
                  // input chunk x has now been read for the last time: the epilogue may overwrite it with output chunk x
                  uint32_t m = (info >> 26) & 0xfu;
                  while (m) { const int x = __ffs((int)m) - 1; m &= m - 1u; umma_commit<CG>(afree_bar0 + 8u * x); }
                }
              }
              __syncwarp();
#if CFN_TC_ISSUE_STAMPS
              prof.stamp();      // diagnostic build: after the issue block
#endif
              cur_full = next_full;
              if (nstage == 0) b_lo = b_lo0; else b_lo += b_step;
              stage = nstage; phase = nphase;
            }
            if (split && pi == 0) {     // the first part's accumulator is complete: its drain starts now
              if (elect_one()) umma_commit<CG>(bar_local(&bars->acc_full));
              __syncwarp();
            }
          }
          if (elect_one()) umma_commit<CG>(bar_local(split ? &bars->acc_full2 : &bars->acc_full));
          __syncwarp();
          prof.stamp();
          if (st.kind == 2) { pending_out = true; ++out_cnt; } else { ++act_gen; ready_upto = 0; }
        }
      }
    }
  } else if (warp == TC_W_WATCH) {
    // profiling only: time at which each stage's TMA data has landed (independent of the MMA thread's progress)
    if (a.prof && blockIdx.x == 0 && rank == 0) {
      int stage = 0; uint32_t phase = 0;
      Prof prof{lane == 0 ? a.prof + 3 * TC_PROF_N : nullptr, 0};
      for (int64_t unit = unit0; unit < a.n_units; unit += n_grid_units)
        for (int g = 0; g < plan.n_steps; ++g) {
          const int n_blk = plan.steps[g].n_parts * plan.steps[g].n_k;
          for (int blk = 0; blk < n_blk; ++blk) {
            mbar_wait(bar_local(&bars->full[stage]), phase);
            prof.stamp();
            if (++stage == a.stages) { stage = 0; phase ^= 1u; }
          }
        }
    }
  } else if (warp < 8) {
    // ================================= encode + epilogue warps (256 threads) =================================
    const int e = warp, q = warp & 3, hh = e >> 2;
    const int tid_e = threadIdx.x;
    const int row = q * 32 + lane;                         // TMEM lane == row of the tile owned by this thread
    const uint32_t tmem_row = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t acc_cnt = 0, split_cnt = 0;
    Prof prof{(a.prof && blockIdx.x == 0 && warp == 0 && lane == 0) ? a.prof : nullptr, 0};
    Prof prof2{nullptr, 0};   // (role 3 of the profile buffer is used by the TMA-landing watcher in warp 3)
    float* sbias = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + sizeof(TcBarriers));   // 512 floats
    auto epi_sync = [&]() { asm volatile("bar.sync 1, 256;" ::: "memory"); };
    // stage the fp32 bias (and tanh flags) of step g into shared memory: read back as warp-wide broadcasts
    auto load_bias = [&](int g) {
      const TcStep& st = plan.steps[g];
      if (st.kind != 2) return;      // hidden layers carry their bias inside the GEMM (ones columns of gamma(d))
      for (int i = tid_e; i < 2 * st.n_total; i += 256) sbias[i] = __ldg(a.table + st.bias_off + i);
    };
    // positional encoding of this thread's row of tile `unit` straight into the swizzled A tiles
    auto encode_tile = [&](int64_t unit) {
      const int64_t m = (unit * CG + rank) * 128 + row;
      const bool valid = m < a.M;
      const int64_t b = valid ? (m / a.N) : 0;
      if (hh != 0) return;          // gamma(d) follows later (encode_gd), into the same tile
      float px = 0.f, py = 0.f, pz = 0.f;
      if (valid) {
        if (a.pts) { px = a.pts[m * 3 + 0]; py = a.pts[m * 3 + 1]; pz = a.pts[m * 3 + 2]; }
        else {
          const float* r = a.rays + b * 11; const float z = a.z_vals[m];
          px = __fadd_rn(r[0], __fmul_rn(r[3], z)); py = __fadd_rn(r[1], __fmul_rn(r[4], z)); pz = __fadd_rn(r[2], __fmul_rn(r[5], z));
        }
      }
      encode_row<FP16, false>(px, py, pz, a.L_pos, gp_base, row);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(bar_leader(&bars->in_ready));
    };
    // gamma(d) of this thread's row over columns 0..31 of the gamma tile, once the last reader of gamma(p) is done
    auto encode_gd = [&](int64_t unit) {
      if (hh != 1) return;
      const int64_t m = (unit * CG + rank) * 128 + row;
      float dx = 0.f, dy = 0.f, dz = 0.f;
      if (m < a.M) {
        const float* vd = a.viewdirs ? (a.viewdirs + (m / a.N) * 3) : (a.rays + (m / a.N) * 11 + 8);
        dx = vd[0]; dy = vd[1]; dz = vd[2];
      }
      encode_row<FP16, true>(dx, dy, dz, a.L_dir, gp_base, row);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(bar_leader(&bars->gd_ready));
    };
    // the gamma tile is last read by the view layer (gamma(d) and the bias column): once that accumulator is complete
    // the NEXT tile's gamma(p) is encoded while the last (small) GEMM of this tile runs
    const int enc_step = plan.n_steps - 2;
    if (unit0 < a.n_units) { load_bias(0); encode_tile(unit0); }
    for (int64_t unit = unit0; unit < a.n_units; unit += n_grid_units) {
      prof.stamp();
      const int64_t m = (unit * CG + rank) * 128 + row;    // global point index of this row
      const bool valid = m < a.M;
      prof.stamp();
      for (int g = 0; g < plan.n_steps; ++g) {
        const TcStep& st = plan.steps[g];
        mbar_wait(bar_local(&bars->acc_full), acc_cnt & 1u); ++acc_cnt;
        prof.stamp();
        tc_fence_after();
        if (st.kind == 2) {
          prof2.stamp();
          epi_sync();                                 // this step's bias / flags are in shared memory
          prof2.stamp();
          // 16-column groups alternate between the two warps of a lane quarter; TMEM is released as soon as the
          // values are in registers, the tanh / stores happen afterwards
          uint32_t v[2][16];
          const int n_grp = st.n_total / 16;
          float* out = a.flow_params + m * a.PP + st.out_col;
          const float* flags = sbias + st.n_total;
          // the last step stages its outputs in the (now free) upper half of the activation tile so that the record
          // rows leave the SM as contiguous, coalesced stores instead of 32 scattered sectors per instruction
          const bool staged = plan.stage_out && g == plan.n_steps - 1;
          const int ld_stage = st.n_valid + 1;
          float* stg = reinterpret_cast<float*>(smem_gen + (size_t)(act_chunks / 2) * TC_CHUNK_BYTES);
          auto emit = [&](int c, float o) {
            if (c < st.n_valid) {
              if (staged) stg[row * ld_stage + c] = o;
              else if (valid) out[c] = o;
            }
          };
          for (int t = 2; 2 * t + hh < n_grp; ++t) {   // wider outputs than 64 columns (n_flows > 4): plain path
            const int gi = 2 * t + hh;
            if (gi * 16 >= st.n_valid) break;
            uint32_t w[16];
            tmem_ld16(tmem_row + (uint32_t)(gi * 16), w);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int c = gi * 16 + i;
              float o = __uint_as_float(w[i]) + sbias[c];
              if (flags[c] != 0.f) o = tanh_fast(o);
              emit(c, o);
            }
          }
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const int gi = 2 * t + hh;
            if (gi < n_grp && gi * 16 < st.n_valid) tmem_ld16(tmem_row + (uint32_t)(gi * 16), v[t]);
          }
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(bar_leader(&bars->out_done));
          prof2.stamp();
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const int gi = 2 * t + hh;
            if (gi < n_grp && gi * 16 < st.n_valid) {
              // bias and flags first (vector broadcasts), then branch-free math, then the stores: nothing in between
              // can alias, so the sixteen outputs are processed with full instruction-level parallelism
              float bb[16], ff[16], o[16];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float4 b4 = reinterpret_cast<const float4*>(sbias + gi * 16)[i];
                const float4 f4 = reinterpret_cast<const float4*>(flags + gi * 16)[i];
                bb[4 * i] = b4.x; bb[4 * i + 1] = b4.y; bb[4 * i + 2] = b4.z; bb[4 * i + 3] = b4.w;
                ff[4 * i] = f4.x; ff[4 * i + 1] = f4.y; ff[4 * i + 2] = f4.z; ff[4 * i + 3] = f4.w;
              }
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float x = __uint_as_float(v[t][i]) + bb[i];
                o[i] = (ff[i] != 0.f) ? tanh_fast(x) : x;
              }
              // unstaged rows: 16-byte stores where the whole quad is valid (record rows are 16-byte aligned: PP = 18F floats,
              // out_col = 3F) instead of sixteen 4-byte ones
              const bool vec_rows = !staged && ((a.PP | st.out_col) & 3) == 0 && (reinterpret_cast<uintptr_t>(a.flow_params) & 15) == 0;
              if (vec_rows) {
                if (valid) {
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    const int c = gi * 16 + 4 * i;
                    if (c + 3 < st.n_valid) *reinterpret_cast<float4*>(out + c) = make_float4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
                    else {
#pragma unroll
                      for (int j = 0; j < 4; ++j) if (c + j < st.n_valid) out[c + j] = o[4 * i + j];
                    }
                  }
                }
              } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) emit(gi * 16 + i, o[i]);
              }
            }
          }
          prof2.stamp();
          if (staged) {
            epi_sync();
            prof2.stamp();
            const int64_t m0 = (unit * CG + rank) * 128;
            const int nv = st.n_valid;
            // one warp per record row, four rows per batch: all shared-memory reads first, then contiguous stores
            for (int r0 = e; r0 < 128; r0 += 32) {
              float val[4][4];
#pragma unroll
              for (int k = 0; k < 4; ++k)
#pragma unroll
                for (int q2 = 0; q2 < 4; ++q2) {
                  const int c = lane + 32 * q2;
                  val[k][q2] = (c < nv) ? stg[(r0 + 8 * k) * ld_stage + c] : 0.f;
                }
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const int r = r0 + 8 * k;
                if (m0 + r < a.M) {
                  float* dst = a.flow_params + (m0 + r) * a.PP + st.out_col;
#pragma unroll
                  for (int q2 = 0; q2 < 4; ++q2) {
                    const int c = lane + 32 * q2;
                    if (c < nv) dst[c] = val[k][q2];
                  }
                }
              }
            }
          }
          prof2.stamp();
        } else {
          const int n_out_chunks = st.n_total / 64;
          // software pipeline over this warp's (chunk, half) pieces: the next TMEM load is in flight while the
          // current 32 columns are biased, activated, packed and stored
          uint32_t va[32], vb[32];
          // (the ReLU decision is taken ONCE per 32-column piece from a register: tested per 8 columns through the
          // schedule in the parameter bank it was an indexed constant load and a branch in front of every store)
          const bool relu = st.kind == 0;
          auto process = [&](uint32_t (&v)[32], int j, int half) {
            const uint32_t chunk = act_base + j * TC_CHUNK_BYTES;
            uint32_t pk[16];
            if (relu) {
#pragma unroll
              for (int i = 0; i < 16; ++i) pk[i] = pack2<FP16, true>(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) pk[i] = pack2<FP16, false>(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
              asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};"
                           :: "r"(chunk + swz(row, half * 4 + u)), "r"(pk[4 * u]), "r"(pk[4 * u + 1]), "r"(pk[4 * u + 2]), "r"(pk[4 * u + 3])
                           : "memory");
          };
          // chunks [j0, j1) of this warp's parity; wait_free: output chunk j overwrites input chunk j, which the second
          // part's MMAs may still be reading (split-commit steps)
          auto drain = [&](int j0, int j1, bool wait_free) {
            const int j_end = j1 < n_out_chunks ? j1 : n_out_chunks;
            if (j0 < j_end) tmem_ld32(tmem_row + (uint32_t)(j0 * 64), va);
            for (int j = j0; j < j1; j += 2) {
              if (j < n_out_chunks) {
                tmem_ld_wait();                                                          // va = (j, half 0)
                tmem_ld32(tmem_row + (uint32_t)(j * 64 + 32), vb);
                if (wait_free) mbar_wait(bar_local(&bars->a_free[j]), split_cnt & 1u);
                process(va, j, 0);
                tmem_ld_wait();                                                          // vb = (j, half 1)
                if (j + 2 < j_end) tmem_ld32(tmem_row + (uint32_t)((j + 2) * 64), va);
                process(vb, j, 1);
                fence_proxy_async();   // generic-proxy stores -> visible to the tensor core's async-proxy reads
                tc_fence_before();
              }
              __syncwarp();
              if (lane == 0) mbar_arrive_cluster(bar_leader(&bars->act_ready[j]));
            }
          };
          if (st.split_commit) {
            const int n_first = st.n_part / 64;      // even: the warp keeps its chunk parity across the two parts
            drain(hh, n_first, true);
            mbar_wait(bar_local(&bars->acc_full2), split_cnt & 1u);              // the second part's accumulator
            tc_fence_after();
            drain(n_first + hh, act_chunks, false);
            ++split_cnt;
          } else {
            drain(hh, act_chunks, false);
          }
        }
        if (st.kind == 2) epi_sync();                 // everyone is done with this step's bias (and the staged outputs)
        {
          const int gn = (g + 1 < plan.n_steps) ? g + 1 : 0;
          if (gn != 0 || unit + n_grid_units < a.n_units) load_bias(gn);
        }
        if (g == plan.gd_step) encode_gd(unit);       // this step's accumulator is complete: gamma(p) is dead
        if (g == enc_step && unit + n_grid_units < a.n_units) encode_tile(unit + n_grid_units);
        prof.stamp();
      }
    }
  }

  // teardown: everything issued has been consumed (the epilogue waited for the last commit)
  tc_fence_before();
  cluster_sync_all();
  if (warp == TC_W_ALLOC) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(512) : "memory");
}

// ======================================================================================================
// weight stream packing
// ======================================================================================================
struct PackSrc { const float* ptr; int ld; };
struct PackSrcTable { PackSrc s[64]; };

// one CUDA block per stream block: [rows_padded][64] 2-byte elements, zero padded
template <bool FP16>
__global__ void pack_stream_kernel(PackSrcTable srcs, const int* __restrict__ blocks, uint16_t* __restrict__ stream) {
  const int* b = blocks + blockIdx.x * 10;
  const int src = b[0], row0 = b[1], rows_valid = b[2], col0 = b[3], cols_valid = b[4], rows_padded = b[5];
  const int64_t stream_row = ((int64_t)(uint32_t)b[7] << 31) | (uint32_t)b[6];
  const int bias_src = b[8], bias_col = b[9];
  const PackSrc S = srcs.s[src];
  for (int i = threadIdx.x; i < rows_padded * 64; i += blockDim.x) {
    const int r = i >> 6, c = i & 63;
    float v = 0.f;
    if (r < rows_valid && c < cols_valid) v = S.ptr[(int64_t)(row0 + r) * S.ld + col0 + c];
    // the bias row multiplies the ones column of the gamma tile; like every weight it is rounded to the operand type
    // (scripts/experiments/k1_precision_sim.py: 3.9e-4 -> 4.0e-4 on the stressed fixture)
    if (bias_src >= 0 && c == bias_col && r < rows_valid) v = srcs.s[bias_src].ptr[row0 + r];
    uint16_t o;
    if (FP16) o = __half_as_ushort(__float2half_rn(fminf(fmaxf(v, -65504.0f), 65504.0f)));   // saturate, never inf
    else o = __bfloat16_as_ushort(__float2bfloat16_rn(v));
    stream[(stream_row + r) * 64 + c] = o;
  }
}

// bias table: table[off + i] = (i < n_valid) ? src[i] : 0
__global__ void pack_bias_kernel(const float* __restrict__ src, float* __restrict__ dst, int n_valid, int n_padded) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_padded) dst[i] = (i < n_valid) ? src[i] : 0.f;
}

// composed bias: out[r] = sum_k am[r,k] * hb[k] + ab[r]
__global__ void compose_bias_kernel(const float* __restrict__ am, const float* __restrict__ hb, const float* __restrict__ ab,
                                    float* __restrict__ out, int rows, int k) {
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  float s = 0.f;
  for (int i = 0; i < k; ++i) s = fmaf(am[r * k + i], hb[i], s);
  out[r] = s + ab[r];
}

// ======================================================================================================
// host side
// ======================================================================================================
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_tensor_map(CUtensorMap* map, void* base, int64_t rows, int box_rows, bool fp16, int box_cols = 64) {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    CFN_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    if (!p || q != cudaDriverEntryPointSuccess) { set_error("cuTensorMapEncodeTiled not available from the driver"); return CFN_ECUDA; }
    fn = (EncodeTiledFn)p;
  }
  cuuint64_t gdim[2] = {64, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {128};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_32B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return CFN_ECUDA; }
  return CFN_OK;
}

// source ids for the pack recipe
enum { SRC_COMP_A_B = 60, SRC_COMP_C_B = 61, SRC_COMP_A = 62, SRC_COMP_C = 63 };   // 0..59: parameter slot index

int tc_create(CfnHandle* h) {
  const CfnConfig& c = h->cfg;
  const int W = c.W, F = c.F, D = c.D;
  CFN_CHECK_ARG(W % 64 == 0 && W >= 128 && W <= 512, "tensor-core path: netwidth %d unsupported (multiple of 64 in 128..512)", W);
  CFN_CHECK_ARG(h->in_pos <= 63 && h->in_dir <= 32, "tensor-core path: multires %d / multires_views %d unsupported (<=10 / <=4)", c.L_pos, c.L_dir);
  CFN_CHECK_ARG(15 * F <= 256, "tensor-core path: n_flows %d unsupported", F);
  CFN_CHECK_ARG(D + 4 <= TC_MAX_STEPS, "tensor-core path: netdepth %d unsupported", D);
  CFN_CHECK_ARG(h->in_dir <= 32, "tensor-core path: multires_views %d unsupported", c.L_dir);
  CFN_CHECK_ARG(h->slots.size() <= 60, "too many parameter tensors");
  TcPlan* p = new TcPlan();
  h->tc = p;
  p->stagger = 0;
  if (const char* e = getenv("CFN_TC_STAGGER")) p->stagger = atoi(e);
  p->prof_dev = nullptr;
  p->stream_dev = nullptr; p->table_dev = nullptr; p->compA = p->compA_b = p->compC = p->compC_b = nullptr; p->blocks_dev = nullptr;
  TcPlanDev& dev = p->dev;
  memset(&dev, 0, sizeof(dev));
  dev.act_chunks = W / 64;
  const int AC = dev.act_chunks;
  int64_t stream_row = 0;
  int table_off = 0;

  struct KCh { int src, kstart, ksteps, col0, cols_valid, with_bias; };
  // every kind 0/1 step multiplies the ones columns (62, 63) of the gamma(d) tile by the (hi, lo) split of its fp32
  // bias, so the epilogue is a pure convert-and-store; kind 2 steps add their (tiny) bias in the epilogue
  auto add_step = [&](int kind, int n_valid, int n_part_max, bool rev, std::vector<KCh> kch, int src_mat, int bias_src,
                      int out_col) {
    TcStep& st = dev.steps[dev.n_steps++];
    st.kind = kind;
    const int gran = 16 * CG;                       // UMMA N granularity (16 per CTA)
    int n_total = ((n_valid + gran - 1) / gran) * gran;
    if (kind != 2) n_total = ((n_valid + 63) / 64) * 64;
    st.n_total = n_total;
    st.n_part = n_total < n_part_max ? n_total : n_part_max;
    st.n_parts = (n_total + st.n_part - 1) / st.n_part;
    st.order_rev = rev ? 1 : 0;
    if (kind != 2) {
      // the bias rides in column 63 of a gamma block if the step reads the gamma tile anyway, else in a K=16 slice of its own
      bool has_g = false;
      for (auto& k : kch)
        if ((k.src == TC_SRC_GD || k.src == TC_SRC_GP) && !has_g) { k.kstart = 0; k.ksteps = 4; k.with_bias = 1; has_g = true; }
      if (!has_g) kch.push_back({TC_SRC_GP, 3, 1, 0, 0, 2});   // with_bias == 2: stand-alone bias entry (SWIZZLE_32B tile)
    }
    st.n_k = (int)kch.size();
    for (int i = 0; i < st.n_k; ++i) {
      const bool gam = kch[i].src == TC_SRC_GP || kch[i].src == TC_SRC_GD;
      const int idx = gam ? AC : kch[i].src;
      // bits 0..15: offset of the A operand in descriptor units (16 bytes) from the activation tile: chunk + K slice
      st.kinfo[i] = (unsigned)((idx * TC_CHUNK_BYTES + kch[i].kstart * 32) >> 4) | ((unsigned)kch[i].ksteps << 16) |
                    ((unsigned)idx << 20) | ((unsigned)(kch[i].with_bias == 2 ? 1 : 0) << 24) |
                    ((unsigned)(kch[i].src == TC_SRC_GD ? 1 : 0) << 25);
      if (kch[i].src == TC_SRC_GP && kch[i].with_bias != 2) dev.gd_step = dev.n_steps - 1;   // last reader of gamma(p)
    }
    st.split_commit = 0;
    if (kind != 2 && st.n_parts == 2 && !st.order_rev && (st.n_part % 128) == 0 && st.n_part / 64 <= 4) {
      st.split_commit = 1;
      for (int x = 0; x < st.n_part / 64; ++x) {
        int pos = 0;                                  // not read by this step: free right after the first K chunk
        for (int i = 0; i < st.n_k; ++i) if (kch[i].src == x) pos = i;
        st.kinfo[pos] |= 1u << (26 + x);
      }
    }
    st.bias_off = table_off;
    st.out_col = out_col;
    st.n_valid = n_valid;
    st.row0 = (int)stream_row;
    // stream blocks in the order the producer consumes them: issue-order parts, then K chunks
    for (int pi = 0; pi < st.n_parts; ++pi) {
      const int pp = st.order_rev ? (st.n_parts - 1 - pi) : pi;
      for (int i = 0; i < st.n_k; ++i) {
        TcPlan::Block b;
        b.src = src_mat;
        b.row0 = pp * st.n_part;
        b.rows_valid = std::max(0, std::min(st.n_part, n_valid - b.row0));
        b.col0 = kch[i].col0;
        b.cols_valid = kch[i].cols_valid;
        b.rows_padded = st.n_part;
        b.stream_row = stream_row;
        b.bias_src = kch[i].with_bias ? bias_src : -1;
        b.bias_col = kch[i].with_bias == 2 ? 15 : 63;   // stand-alone tile: K slice 48..63 -> tile columns 0..15
        p->blocks.push_back(b);
        stream_row += st.n_part;
      }
    }
    if (kind == 2) {
      TcPlan::BiasSeg bs{bias_src, n_valid, n_total, table_off, 1, out_col};
      p->bias_segs.push_back(bs);
      table_off += 2 * n_total;
    }
  };

  // trunk
  for (int i = 0; i < D; ++i) {
    std::vector<KCh> kch;
    const int slot = h->s_pts(i, 0);
    if (i == 0) kch.push_back({TC_SRC_GP, 0, 4, 0, h->in_pos, 0});
    else if (h->skip >= 0 && i == h->skip + 1) {
      kch.push_back({TC_SRC_GP, 0, 4, 0, h->in_pos, 0});                                      // cat[gamma(p), h] (models.py:171-172)
      for (int j = 0; j < AC; ++j) kch.push_back({j, 0, 4, h->in_pos + 64 * j, 64, 0});
    } else {
      for (int j = 0; j < AC; ++j) kch.push_back({j, 0, 4, 64 * j, 64, 0});
    }
    add_step(0, W, 256, false, kch, slot, slot + 1, 0);
  }
  // composed alpha conditioning from h7 (N = 3F), then the feature layer (parts reversed so that the drain of
  // TMEM columns 0..63 by the alpha epilogue overlaps the first feature MMAs)
  {
    std::vector<KCh> kch;
    for (int j = 0; j < AC; ++j) kch.push_back({j, 0, 4, 64 * j, 64, 0});
    add_step(2, 3 * F, 256, false, kch, SRC_COMP_A, SRC_COMP_A_B, 0);
    add_step(1, W, 256, true, kch, h->s_feat, h->s_feat + 1, 0);
    // view layer on cat[feature, gamma(d)] (models.py:177-181); its gamma(d) block also carries the bias columns
    kch.push_back({TC_SRC_GD, 0, 4, W, h->in_dir, 1});
    add_step(0, W / 2, 256, false, kch, h->s_views, h->s_views + 1, 0);
  }
  // composed rgb conditioning from the view features (N = 15F)
  {
    std::vector<KCh> kch;
    for (int j = 0; j < (W / 2 + 63) / 64; ++j) {
      const int cols = std::min(64, W / 2 - 64 * j);
      kch.push_back({j, 0, cols / 16, 64 * j, cols, 0});
    }
    add_step(2, 15 * F, 256, false, kch, SRC_COMP_C, SRC_COMP_C_B, 3 * F);
  }
  // staging the last step's record rows needs 128 x (15F+1) floats in the upper half of the activation tile
  dev.stage_out = ((size_t)128 * (15 * F + 1) * sizeof(float) <= (size_t)(AC - AC / 2) * TC_CHUNK_BYTES) ? 1 : 0;
  p->stream_rows = stream_row;
  p->table_floats = table_off;

  cudaDeviceProp prop;
  int devid = 0;
  auto fail = [&](const char* what) { set_error("tc_create: %s", what); return CFN_ECUDA; };
  if (cudaGetDevice(&devid) != cudaSuccess || cudaGetDeviceProperties(&prop, devid) != cudaSuccess) return fail("device query");
  if (prop.major != 10) { set_error("tensor-core path needs sm_100 (found sm_%d%d)", prop.major, prop.minor); return CFN_EINVAL; }
  p->num_sms = prop.multiProcessorCount;
  p->stage_bytes = (256 / CG) * 128;
  const size_t fixed = (size_t)(AC + 1) * TC_CHUNK_BYTES + sizeof(TcBarriers) + 2048;   // + bias staging (512 floats)
  const size_t smem_max = (size_t)prop.sharedMemPerBlockOptin;
  int stages = (int)((smem_max - fixed) / p->stage_bytes);
  if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
  if (stages < 2) return fail("not enough shared memory for two weight stages");
  p->stages = stages;
  p->smem_bytes = fixed + (size_t)stages * p->stage_bytes;

  if (getenv("CFN_TC_PROFILE")) {
    if (cudaMalloc(&p->prof_dev, 4 * TC_PROF_N * sizeof(unsigned long long)) != cudaSuccess) return fail("cudaMalloc(prof)");
    cudaMemset(p->prof_dev, 0, 4 * TC_PROF_N * sizeof(unsigned long long));
  }
  if (cudaMalloc(&p->stream_dev, (size_t)p->stream_rows * 128) != cudaSuccess) return fail("cudaMalloc(stream)");
  if (cudaMalloc(&p->table_dev, (size_t)p->table_floats * sizeof(float)) != cudaSuccess) return fail("cudaMalloc(table)");
  if (cudaMalloc(&p->compA, (size_t)3 * F * W * sizeof(float)) != cudaSuccess) return fail("cudaMalloc");
  if (cudaMalloc(&p->compA_b, (size_t)3 * F * sizeof(float)) != cudaSuccess) return fail("cudaMalloc");
  if (cudaMalloc(&p->compC, (size_t)15 * F * (W / 2) * sizeof(float)) != cudaSuccess) return fail("cudaMalloc");
  if (cudaMalloc(&p->compC_b, (size_t)15 * F * sizeof(float)) != cudaSuccess) return fail("cudaMalloc");
  std::vector<int> flat;
  for (auto& b : p->blocks) {
    flat.push_back(b.src); flat.push_back(b.row0); flat.push_back(b.rows_valid); flat.push_back(b.col0);
    flat.push_back(b.cols_valid); flat.push_back(b.rows_padded);
    flat.push_back((int)(b.stream_row & 0x7FFFFFFF)); flat.push_back((int)(b.stream_row >> 31));
    flat.push_back(b.bias_src); flat.push_back(b.bias_col);
  }
  if (cudaMalloc(&p->blocks_dev, flat.size() * sizeof(int)) != cudaSuccess) return fail("cudaMalloc(blocks)");
  if (cudaMemcpy(p->blocks_dev, flat.data(), flat.size() * sizeof(int), cudaMemcpyHostToDevice) != cudaSuccess) return fail("cudaMemcpy(blocks)");
  if (cudaMemset(p->table_dev, 0, (size_t)p->table_floats * sizeof(float)) != cudaSuccess) return fail("cudaMemset");
  // tanh flags of the two output steps never change
  for (auto& bs : p->bias_segs) {
    if (!bs.with_flags) continue;
    if (cudaMemcpy(p->table_dev + bs.off + bs.n_padded, h->tanh_flags + bs.flag_off, (size_t)bs.n_valid * sizeof(float),
                   cudaMemcpyDeviceToDevice) != cudaSuccess) return fail("cudaMemcpy(flags)");
  }
  const bool fp16 = c.precision == CFN_PREC_FP16;
  int rc;
  if ((rc = make_tensor_map(&p->tm_big, p->stream_dev, p->stream_rows, 128, fp16))) return rc;
  if ((rc = make_tensor_map(&p->tm_small, p->stream_dev, p->stream_rows, 16, fp16))) return rc;
  if ((rc = make_tensor_map(&p->tm_bias, p->stream_dev, p->stream_rows, 128, fp16, 16))) return rc;   // [128 rows][16 cols], SWIZZLE_32B
  auto set_attr = [&](const void* fnp) {
    return cudaFuncSetAttribute(fnp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem_bytes) == cudaSuccess;
  };
  const bool ok = fp16 ? set_attr((const void*)mlp_tc_kernel<true>) : set_attr((const void*)mlp_tc_kernel<false>);
  if (!ok) return fail("cudaFuncSetAttribute(max dynamic shared memory)");
  return CFN_OK;
}

void tc_destroy(CfnHandle* h) {
  TcPlan* p = h->tc;
  if (!p) return;
  cudaFree(p->stream_dev); cudaFree(p->table_dev); cudaFree(p->compA); cudaFree(p->compA_b); cudaFree(p->compC);
  cudaFree(p->compC_b); cudaFree(p->blocks_dev); cudaFree(p->prof_dev);
  delete p;
  h->tc = nullptr;
}

int tc_pack(CfnHandle* h, cudaStream_t s) {
  TcPlan* p = h->tc;
  const CfnConfig& c = h->cfg;
  const int W = c.W, F = c.F;
  int rc;
  // compose: compA (3F x W) = amA (3F x h_alpha) . W_halpha (h_alpha x W);  bias = amA . b_halpha + amA_b
  {
    GemmArgs g{};
    g.A = h->amA; g.a_rs = c.h_alpha; g.a_cs = 1;
    g.B = h->w32 + h->slots[h->s_halpha].offset; g.b_rs = W; g.b_cs = 1;
    g.C = p->compA; g.c_rs = W; g.M = 3 * F; g.N = W; g.K = c.h_alpha; g.split_k = 1;
    if ((rc = launch_sgemm(g, s))) return rc;
    compose_bias_kernel<<<1, 128, 0, s>>>(h->amA, h->w32 + h->slots[h->s_halpha + 1].offset, h->amA_b, p->compA_b, 3 * F, c.h_alpha);
    g.A = h->amC; g.a_rs = c.h_rgb;
    g.B = h->w32 + h->slots[h->s_hrgb].offset; g.b_rs = W / 2;
    g.C = p->compC; g.c_rs = W / 2; g.M = 15 * F; g.N = W / 2; g.K = c.h_rgb;
    if ((rc = launch_sgemm(g, s))) return rc;
    compose_bias_kernel<<<1, 128, 0, s>>>(h->amC, h->w32 + h->slots[h->s_hrgb + 1].offset, h->amC_b, p->compC_b, 15 * F, c.h_rgb);
    CFN_LAUNCH_CHECK();
  }
  PackSrcTable t;
  memset(&t, 0, sizeof(t));
  for (size_t i = 0; i < h->slots.size(); ++i) { t.s[i].ptr = h->w32 + h->slots[i].offset; t.s[i].ld = h->slots[i].cols; }
  t.s[SRC_COMP_A] = {p->compA, W};
  t.s[SRC_COMP_C] = {p->compC, W / 2};
  t.s[SRC_COMP_A_B] = {p->compA_b, 1};
  t.s[SRC_COMP_C_B] = {p->compC_b, 1};
  const bool fp16 = c.precision == CFN_PREC_FP16;
  if (fp16) pack_stream_kernel<true><<<(unsigned)p->blocks.size(), 256, 0, s>>>(t, p->blocks_dev, (uint16_t*)p->stream_dev);
  else pack_stream_kernel<false><<<(unsigned)p->blocks.size(), 256, 0, s>>>(t, p->blocks_dev, (uint16_t*)p->stream_dev);
  CFN_LAUNCH_CHECK();
  for (auto& bs : p->bias_segs) {
    const float* src = bs.src == SRC_COMP_A_B ? p->compA_b : (bs.src == SRC_COMP_C_B ? p->compC_b : h->w32 + h->slots[bs.src].offset);
    pack_bias_kernel<<<(bs.n_padded + 127) / 128, 128, 0, s>>>(src, p->table_dev + bs.off, bs.n_valid, bs.n_padded);
  }
  CFN_LAUNCH_CHECK();
  return CFN_OK;
}

size_t tc_workspace_bytes(const CfnHandle*, int64_t) { return 256; }

int tc_debug_profile(CfnHandle* h, unsigned long long* out_host, int n) {
  TcPlan* p = h->tc;
  if (!p || !p->prof_dev) { set_error("profiling buffer not enabled (set CFN_TC_PROFILE=1 before cfn_create)"); return CFN_ESTATE; }
  if (n > 4 * TC_PROF_N) n = 4 * TC_PROF_N;
  CFN_CUDA(cudaDeviceSynchronize());
  CFN_CUDA(cudaMemcpy(out_host, p->prof_dev, (size_t)n * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return CFN_OK;
}

int tc_network_fwd(CfnHandle* h, const float* rays, const float* z_vals, const float* pts, const float* viewdirs,
                   int64_t B, int N, float* flow_params, void*, size_t, cudaStream_t s) {
  TcPlan* p = h->tc;
  TcArgs a;
  a.rays = rays; a.z_vals = z_vals; a.pts = pts; a.viewdirs = viewdirs;
  a.M = B * N; a.N = N; a.L_pos = h->cfg.L_pos; a.L_dir = h->cfg.L_dir;
  a.table = p->table_dev; a.flow_params = flow_params; a.PP = h->PP;
  a.n_units = (a.M + 128 * CG - 1) / (128 * CG);
  a.stages = p->stages; a.stage_bytes = p->stage_bytes;
  a.prof = p->prof_dev;
  a.stagger = p->stagger;
  int64_t units_grid = p->num_sms / CG;
  if (units_grid > a.n_units) units_grid = a.n_units;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(units_grid * CG));
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = p->smem_bytes;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  const bool fp16 = h->cfg.precision == CFN_PREC_FP16;
  const cudaError_t e = fp16 ? cudaLaunchKernelEx(&cfg, mlp_tc_kernel<true>, p->tm_big, p->tm_small, p->tm_bias, p->dev, a)
                             : cudaLaunchKernelEx(&cfg, mlp_tc_kernel<false>, p->tm_big, p->tm_small, p->tm_bias, p->dev, a);
  if (e != cudaSuccess) { set_error("mlp_tc_kernel launch failed: %s", cudaGetErrorString(e)); return CFN_ECUDA; }
  return CFN_OK;
}

}  // namespace cfn
