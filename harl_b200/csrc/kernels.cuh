// Internal kernel-launcher interface shared by the translation units.
#pragma once
#include "common.cuh"

namespace hb {

enum { MODE_ACT = 0, MODE_EVAL = 1, MODE_GRAD = 2 };

struct HeadArgs {
  const float* feat;     // [rows, h]  trunk output (batch-row indexed)
  int h, out;
  const float* hw;       // [out][h]
  const float* hbias;    // [out]
  const float* log_std;  // [out] (Box)
  float std_x, std_y;
  int64_t rows;
  const int32_t* index;  // batch row -> buffer row (nullable)
  // act
  int deterministic;
  uint64_t seed, offset;
  const unsigned long long* offset_base;  // device counter added to offset inside the kernel (CUDA-graph replays), nullable
  float* actions_out;    // [rows, ad]
  float* logp_out;       // [rows, ad]
  // evaluate / grad (buffer-row indexed)
  const float* actions;
  const float* avail;
  const float* old_logp;
  const float* adv;
  const float* factor;
  const float* active;
  const float* logp_ref;
  float* factor_inout;
  int agg_prod;
  // grad
  float clip, entropy_coef;
  int use_active, use_clip;
  const double* norm3;
  float* dfeat;          // [rows, h]
  float* g_hw;           // [out][h]
  float* g_hbias;        // [out]
  float* g_log_std;      // [out]
  double* scalars;       // += (loss_num, entropy_num, ratio_sum, rows)
  // fused LayerNorm + activation backward of the last trunk block (grad mode, when ln_z != nullptr):
  // dfeat then receives dZ_L instead of d/d features, and the LN affine gradients are accumulated here
  const float* ln_z; const float* ln_stats; const float* ln_w; float* g_ln_w; float* g_ln_b; int ln_act;
  // parameter-gradient sums go to slot blockIdx.x of a split buffer (g_ptr + part_delta + blockIdx.x * part_stride, plain
  // read-modify-write, summed once per call by dw_reduce) instead of same-address global atomics; 0 = atomics
  int64_t part_delta, part_stride;
};

struct ValueArgs {
  const float* feat; int h;
  const float* hw; const float* hbias;
  int64_t rows; const int32_t* index;
  float* values_out;            // forward mode
  const float* value_preds; const float* returns;  // buffer-row indexed
  const float* vn_state;        // nullable
  float clip, huber_delta, coef;  // coef = value_loss_coef * inv_count
  int use_huber, use_clipped;
  float* dfeat; float* g_hw; float* g_hbias; double* scalars;  // scalars += (loss_sum, rows)
  const float* ln_z; const float* ln_stats; const float* ln_w; float* g_ln_w; float* g_ln_b; int ln_act;  // as in HeadArgs
  int64_t part_delta, part_stride;
};

// launchers (gemm_simt.cu, rowwise.cu, optim.cu)
int launch_linear_ln_fwd(int act, const float* X, int ldx, const float* WT, const float* bias, const float* lnw,
                         const float* lnb, float* Z, float* Y, float* stats, int64_t M, int N, int Kred, cudaStream_t st);
int launch_dx_ln_bwd(int act, const float* dZ, int N, const float* W, const float* Zp, const float* stats_p,
                     const float* lnw_p, float* dZp, float* g_lnw_p, float* g_lnb_p, int64_t M, int Np, cudaStream_t st);
int launch_dw_accum(const float* dZ, int N, const float* X, int ldx, int K, float* dW, float* db, int64_t M,
                    cudaStream_t st);
int launch_feat_norm(const float* obs, int in_dim, const int32_t* index, int64_t rows, int feature_norm, float* xout,
                     int ldx, cudaStream_t st);
int launch_ln_act_bwd(const float* dY, const float* Z, const float* stats, const float* lnw, float* dZ, float* g_lnw,
                      float* g_lnb, int64_t rows, int N, int act, cudaStream_t st);
int launch_featnorm_fold(const hb_net_desc* d, const float* params, float* grad, cudaStream_t st);

// tcgen05 3xTF32 layer-wise kernels (tc_gemm.cu)
int launch_tc_linear_ln_fwd(int act, const float* X, int ldx, const float* tiles, int nchunks, const float* bias, const float* lnw, const float* lnb, float* Z, float* Y, float* stats,
                            int64_t M, int N, int Kred, cudaStream_t st);
int launch_tc_dx_ln_bwd(int act, const float* dZ, int N, const float* tiles, int nchunks, const float* Zp,
                        const float* stats_p, const float* lnw_p, float* dZp, float* g_lnw_p, float* g_lnb_p, int64_t M,
                        int Np, int64_t part_delta, int64_t part_stride, cudaStream_t st);
int launch_tc_dw_accum(const float* dZ, int N, const float* X, int ldx, int K, float* dW, float* db,
                       int64_t M, int64_t part_stride, cudaStream_t st);
// tensor-core tangent block, selected by hb_set_trpo_jvp_impl(1) (the default)
int launch_tc_jvp_linear_ln(int act, const float* X, int ldx, const float* Xd, const float* tiles,
                            const float* tiles_d, int nchunks, const float* bd, const float* lnw, const float* lnwd,
                            const float* lnbd, const float* Z, const float* stats, float* Yd, int64_t M, int N, int Kred,
                            cudaStream_t st);
int launch_pack_umma_tiles(const float* W, int ldn, int ldk, const float* scale, int N, int K, int NT, int nchunks,
                           float* dst, cudaStream_t st);
int tc_dw_splits();
int launch_dw_reduce(float* grad, const float* part, int total, cudaStream_t st);

int launch_policy_head(int head, int mode, const HeadArgs& a, cudaStream_t st);
int launch_value_head(int grad, const ValueArgs& a, cudaStream_t st);
// row-group variants for the common widths (heads_fast.cu); *handled = false -> fall back to the generic kernels
int launch_policy_head_rows(int head, int mode, const HeadArgs& a, cudaStream_t st, bool* handled);
int launch_value_head_rows(int grad, const ValueArgs& a, cudaStream_t st, bool* handled);


}  // namespace hb
