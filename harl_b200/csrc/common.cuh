// Shared device/host helpers for the harl_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/harl_b200.h"

namespace hb {

// ------------------------------------------------------------------ error plumbing
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define HB_CHECK_ARG(cond, msg)                          \
  do {                                                   \
    if (!(cond)) {                                       \
      hb::set_error("%s: %s", __func__, msg);            \
      return HB_ERR_INVALID;                             \
    }                                                    \
  } while (0)

// Called right after every kernel launch: error check, launch counter, optional profiling event.
void note_launch(const char* what, cudaStream_t st);
const char* shape_label(const char* base, int64_t m, int n, int k);

#define HB_LAUNCH_DONE(st, what)                         \
  do {                                                   \
    cudaError_t _e = cudaGetLastError();                 \
    if (_e != cudaSuccess) return hb::cuda_fail(_e, what); \
    hb::note_launch(what, st);                           \
  } while (0)

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ------------------------------------------------------------------ derived-weight layout
// "prepared" buffer: what the forward kernels read.  For trunk layer l (0-based):
//   wt[l]   : [kpad_l][n_l]  W^T with the feature-norm gamma folded into layer 0
//   bias[l] : [n_l]          (layer 0: b + W beta0 when feature_norm)
//   lnw[l], lnb[l] : [n_l]
// head: hw [out][h], hb [out], log_std [out] (Box), copied verbatim.
struct PrepLayout {
  int n_layers;
  int k[HB_MAX_LAYERS], kpad[HB_MAX_LAYERS], n[HB_MAX_LAYERS];
  int wt[HB_MAX_LAYERS], bias[HB_MAX_LAYERS], lnw[HB_MAX_LAYERS], lnb[HB_MAX_LAYERS];
  int hw, hbias, log_std;
  // GRU (rnn.py:8-81), rnn_layers > 0: per layer W_ih^T and W_hh^T as [h][3h] (gate order r, z, n), the two bias
  // vectors [3h], then the output LayerNorm affine
  int rnn_layers, rh;
  int rnn_wih_t[2], rnn_whh_t[2], rnn_bih[2], rnn_bhh[2], rnn_lnw, rnn_lnb;
  // tcgen05 operand images (tc_gemm.cu): per layer, per 32-wide k-chunk: hi image [nt][32] then lo image
  int tk[HB_MAX_LAYERS], tk_chunks[HB_MAX_LAYERS], tk_nt[HB_MAX_LAYERS];
  // images of W^T for the backward dX GEMM (layers >= 1)
  int tkt[HB_MAX_LAYERS], tkt_chunks[HB_MAX_LAYERS], tkt_nt[HB_MAX_LAYERS];
  // fused update kernel (fused_update.cu): fp16 hi/lo operand images of the LayerNorm-affine-folded weights
  //   W'_l = W_l diag(gamma_{l-1}),  b'_l = b_l + W_l beta_{l-1}   (gamma_{-1}, beta_{-1} = the feature-norm affine)
  // per layer, per 32-wide k-chunk (the last may be 16 wide): hi image [n_l][kc] then lo image, K-major no-swizzle core
  // matrices; the head likewise as one [16][h] image pair.  fz_ok = 0: shape outside the fused kernel (layer-wise path).
  int fz_ok, fz_k0p;
  int fz_w[2], fz_chunks[2], fz_bias[2];
  int fz_w1b;                        // layer 1 again, chunked by 32 OUTPUT rows ([32][h] images): the dX GEMM's B operand
  int fz_hw, fz_hbias, fz_scale;
  int total;
};

// Offsets into the flat parameter buffer (reference state_dict order).
struct ParamLayout {
  int fn_w, fn_b;  // feature norm (-1 if absent)
  int w[HB_MAX_LAYERS], b[HB_MAX_LAYERS], lnw[HB_MAX_LAYERS], lnb[HB_MAX_LAYERS];
  int hw, hbias, log_std;  // head
  int rnn_wih[2], rnn_whh[2], rnn_bih[2], rnn_bhh[2], rnn_lnw, rnn_lnb;  // GRU [3h][h] x2, [3h] x2 per layer; LN
  int total;
};

int make_layouts(const hb_net_desc* d, ParamLayout* pl, PrepLayout* pp, hb_net_layout* out);
int gemm_impl();  // 0 = FP32 SIMT, 1 = tcgen05 3xTF32 (fp32-accurate)

// ------------------------------------------------------------------ device helpers
#ifdef __CUDACC__

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// sum across the 16 lanes of a half-warp (lanes sharing lane/16)
__device__ __forceinline__ float half_warp_sum(float v) {
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int ACT>
__device__ __forceinline__ float act_fwd(float z) {
  if (ACT == HB_ACT_RELU) return fmaxf(z, 0.f);
  if (ACT == HB_ACT_TANH) return tanhf(z);
  if (ACT == HB_ACT_SIGMOID) return 1.f / (1.f + expf(-z));
  if (ACT == HB_ACT_LEAKY_RELU) return z > 0.f ? z : 0.01f * z;
  if (ACT == HB_ACT_SELU) {
    const float a = 1.6732632423543772848170429916717f, s = 1.0507009873554804934193349852946f;
    return s * (z > 0.f ? z : a * (expf(z) - 1.f));
  }
  if (ACT == HB_ACT_HARDSWISH) return z * fminf(fmaxf(z + 3.f, 0.f), 6.f) / 6.f;
  return z;
}
// d act / dz given the pre-activation z
template <int ACT>
__device__ __forceinline__ float act_bwd(float z) {
  if (ACT == HB_ACT_RELU) return z > 0.f ? 1.f : 0.f;
  if (ACT == HB_ACT_TANH) { float t = tanhf(z); return 1.f - t * t; }
  if (ACT == HB_ACT_SIGMOID) { float s = 1.f / (1.f + expf(-z)); return s * (1.f - s); }
  if (ACT == HB_ACT_LEAKY_RELU) return z > 0.f ? 1.f : 0.01f;
  if (ACT == HB_ACT_SELU) {
    const float a = 1.6732632423543772848170429916717f, s = 1.0507009873554804934193349852946f;
    return z > 0.f ? s : s * a * expf(z);
  }
  if (ACT == HB_ACT_HARDSWISH) return z < -3.f ? 0.f : (z > 3.f ? 1.f : (2.f * z + 3.f) / 6.f);
  return 1.f;
}
__device__ __forceinline__ float act_fwd_rt(int act, float z) {
  switch (act) {
    case HB_ACT_RELU: return act_fwd<HB_ACT_RELU>(z);
    case HB_ACT_TANH: return act_fwd<HB_ACT_TANH>(z);
    case HB_ACT_SIGMOID: return act_fwd<HB_ACT_SIGMOID>(z);
    case HB_ACT_LEAKY_RELU: return act_fwd<HB_ACT_LEAKY_RELU>(z);
    case HB_ACT_SELU: return act_fwd<HB_ACT_SELU>(z);
    case HB_ACT_HARDSWISH: return act_fwd<HB_ACT_HARDSWISH>(z);
    default: return z;
  }
}
__device__ __forceinline__ float act_bwd_rt(int act, float z) {
  switch (act) {
    case HB_ACT_RELU: return act_bwd<HB_ACT_RELU>(z);
    case HB_ACT_TANH: return act_bwd<HB_ACT_TANH>(z);
    case HB_ACT_SIGMOID: return act_bwd<HB_ACT_SIGMOID>(z);
    case HB_ACT_LEAKY_RELU: return act_bwd<HB_ACT_LEAKY_RELU>(z);
    case HB_ACT_SELU: return act_bwd<HB_ACT_SELU>(z);
    case HB_ACT_HARDSWISH: return act_bwd<HB_ACT_HARDSWISH>(z);
    default: return 1.f;
  }
}

// ValueNorm denormalisation of the returns kernels (valuenorm.py:38-45,78-92), every operation separately rounded as
// in the reference: V^ = v * sqrt(max(E[v^2] - E[v]^2, 1e-2)) + E[v] with E[.] = running sum / max(debiasing term,
// 1e-5).  vn == nullptr: no ValueNorm, V^ = v.
struct VNConst { float mean, std; int on; };

__device__ __forceinline__ VNConst vn_load(const float* __restrict__ vn) {
  VNConst c;
  c.on = vn != nullptr;
  c.mean = 0.f;
  c.std = 1.f;
  if (c.on) {
    float d = fmaxf(vn[2], 1e-5f);
    float m = __fdiv_rn(vn[0], d), msq = __fdiv_rn(vn[1], d);
    float var = fmaxf(__fsub_rn(msq, __fmul_rn(m, m)), 1e-2f);
    c.mean = m;
    c.std = __fsqrt_rn(var);
  }
  return c;
}
__device__ __forceinline__ float denorm(const VNConst& c, float v) {
  return c.on ? __fadd_rn(__fmul_rn(v, c.std), c.mean) : v;
}

// gradient-sum output: a fire-and-forget reduction into this CTA's split-buffer slot (slot != 0: a handful of CTAs
// share a slot at most, so no same-address serialisation) or into the gradient itself (slot == 0)
__device__ __forceinline__ void acc_out(float* p, float v, int64_t slot) { atomicAdd(p + slot, v); }

// Philox4x32-10 (Salmon et al. 2011), counter-based: one call -> 4 x 32 random bits.
__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
__device__ __forceinline__ float u01(uint32_t x) {  // (0, 1]
  return ((float)(x >> 8) + 1.0f) * (1.0f / 16777216.0f);
}

#endif  // __CUDACC__
}  // namespace hb
