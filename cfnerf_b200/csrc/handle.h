// Handle layout shared by the C-ABI translation units.
#pragma once
#include <string>
#include <vector>

#include "common.cuh"

struct GatherRow {
  int slot_w;   // parameter slot of the source weight matrix
  int slot_b;   // parameter slot of the source bias
  int row;      // row of the source nn.Linear
  int tanh;     // 1: the reference applies tanh to this output (amor_diag1/2, models.py:367-368)
};

struct ParamSlot {
  std::string name;
  int64_t numel;
  int rows, cols;     // nn.Linear weight (rows=out, cols=in); bias/globals: rows=numel, cols=1
  int64_t offset;     // float offset inside w32
};

// GEMM-operand view of an nn.Linear weight: row stride padded to a multiple of 4 floats (TMA needs 16-byte strides) and,
// for the skip layer, a gap after the gamma(p) columns so that the h columns start 16-byte aligned:
// original column c lives at c + (c >= gap_at ? gap : 0); pad columns are zero.
struct WView {
  const float* p;
  int ld, gap_at, gap;
};

namespace cfn { struct TcPlan; }  // tensor-core weight stream + launch plan (mlp_tc.cu)

struct CfnHandle {
  CfnConfig cfg;
  int in_pos, in_dir, PP, skip;   // skip = index of the layer whose output is concatenated with gamma(p); -1 = none
  std::vector<ParamSlot> slots;
  int64_t n_floats;               // total master floats
  bool packed;

  // slot indices
  int s_pts(int i, int bias) const { return 4 + 2 * i + bias; }
  int s_views, s_feat, s_halpha, s_hrgb, s_frgb, s_falpha;   // base index of each (weight; +1 = bias)

  // device buffers (handle-owned)
  float* w32;        // fp32 copy of every parameter, slot order
  float* globals;    // -> w32 + 0 : alpha_mean, alpha_std, rgb_mean(3), rgb_std(3)
  float* amA;        // (3F, h_alpha) gathered alpha conditioning matrix
  float* amA_b;      // (3F)
  float* amC;        // (15F, h_rgb) gathered rgb conditioning matrix
  float* amC_b;      // (15F)
  float* tanh_flags; // (18F) 1.0 where the output is a tanh'ed diagonal
  int* gatherA_dev;  // (3F,4) GatherRow
  int* gatherC_dev;  // (15F,4)
  std::vector<GatherRow> gatherA, gatherC;

  // GEMM operands of the layer-by-layer network stage (mlp_chain.cu): fp32 FMA (gemm_tc = 0) or tcgen05 kind::tf32
  int gemm_tc;              // 1: contractions run on the tensor cores (every precision mode except CFN_PREC_FP32)
  int chain_bf16;           // 1 (CFN_PREC_BF16): activations, gradients and operand weights of the chain are stored as bf16
                            //   (tcgen05 kind::f16); 0: fp32 storage (kind::tf32 when gemm_tc, fp32 FMA otherwise)
  int gp, gd;               // in_pos / in_dir rounded up to a multiple of 8 (activation / weight column padding)
  float* wg;                // padded operand copy of every weight matrix (tf32-rounded fp32, or bf16 when chain_bf16)
  int64_t wg_floats;
  std::vector<WView> wv;    // per slot (biases: p = nullptr)
  std::vector<int64_t> wg_offset;   // in 4-byte slots
  float* amA_g; float* amC_g;   // operand copies of amA / amC (tf32-rounded when gemm_tc, else aliases)

  // opt-in deterministic weight gradients (cfn_set_deterministic): scratch for the split-K slabs of one wgrad
  int deterministic;
  float* det_scratch; int64_t det_floats;

  cfn::TcPlan* tc;   // nullptr in fp32 mode
  int tc_dirty;      // the fp32 copies changed since K1's weight stream was built (rebuilt lazily by cfn_network_fwd)
};

namespace cfn {
// layer-by-layer chain: check mode, CFN_PREC_TF32 and every training path (mlp_chain.cu)
size_t chain_workspace_floats(const CfnHandle* h, int64_t n_points, int save);
int chain_network_fwd(CfnHandle* h, const float* rays, const float* z_vals, const float* pts, const float* viewdirs,
                     int64_t B, int N, float* flow_params, float* ws, int save, cudaStream_t s);
int chain_network_bwd(const CfnHandle* h, const float* g_flow_params, int64_t B, int N, float* ws, float* const* grads,
                      cudaStream_t s);
int pack_fp32(CfnHandle* h, const float* const* params, cudaStream_t s);

// tensor-core path (mlp_tc.cu)
int tc_create(CfnHandle* h);
void tc_destroy(CfnHandle* h);
int tc_pack(CfnHandle* h, cudaStream_t s);
size_t tc_workspace_bytes(const CfnHandle* h, int64_t n_points);
int tc_debug_profile(CfnHandle* h, unsigned long long* out_host, int n);
int tc_network_fwd(CfnHandle* h, const float* rays, const float* z_vals, const float* pts, const float* viewdirs,
                   int64_t B, int N, float* flow_params, void* ws, size_t ws_bytes, cudaStream_t s);
}  // namespace cfn
