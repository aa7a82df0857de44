// GAE / return scan, advantages, masked moments, ValueNorm (sm_100a).
//
// hb_gae_returns restates OnPolicyCriticBuffer{EP,FP}.compute_returns
// (harl/common/buffers/on_policy_critic_buffer_ep.py:97-200) + the advantage subtraction of
// harl/runners/on_policy_ha_runner.py:26-33, bit-exactly: every multiply / add is separately
// rounded (__fmul_rn/__fadd_rn, no FMA contraction) and the time recurrence is evaluated in
// the reference's order.
//
// HBM-bound: 24 B per (t, column) element.  A CTA stages a [T+1] x CW column tile of the
// four input arrays into shared memory with 16-byte cp.async (all loads in flight at once),
// all threads form V^ = denorm(v) and delta_t in parallel, CW threads run the serial
// recurrence out of shared memory, then all threads write returns/advantages coalesced.
#include "common.cuh"

namespace hb {

// gae_seg.cu
bool launch_gae_seg(const float* rewards, float* value_preds, const float* masks, const float* bad_masks,
                    const float* next_value, float* returns, float* advantages, int T, int64_t C, float gamma, float gl,
                    int ptl, const float* vn, cudaStream_t st, int* rc);

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// ------------------------------------------------------------------ tiled kernel
// smem: vhat [T+1][CW], msk [T+1][CW], bad [T+1][CW], work [T][CW] (rewards -> delta -> gae/returns)
template <int CW>
__global__ void __launch_bounds__(256) gae_tiled_kernel(const float* __restrict__ rewards, float* __restrict__ value_preds,
                                                        const float* __restrict__ masks, const float* __restrict__ bad_masks,
                                                        const float* __restrict__ next_value, float* __restrict__ returns,
                                                        float* __restrict__ adv, int T, int64_t C, float gamma, float gl,
                                                        int use_gae, int ptl, const float* __restrict__ vn) {
  extern __shared__ __align__(16) float sm[];
  float* s_v = sm;
  float* s_m = s_v + (size_t)(T + 1) * CW;
  float* s_b = s_m + (size_t)(T + 1) * CW;
  float* s_w = s_b + (size_t)(T + 1) * CW;
  const int64_t c0 = (int64_t)blockIdx.x * CW;
  const int tid = threadIdx.x;
  const VNConst vc = vn_load(vn);
  // ---- stage: (T+1) rows x CW/4 float4 per array (C % 4 == 0 guaranteed by the launcher), in GAE_CH time chunks
  // issued LAST CHUNK FIRST, one cp.async group each: the backward recurrence starts on the last chunk while the
  // earlier ones are still in flight, and each chunk's results stream out while the next one is being consumed.
  constexpr int V4 = CW / 4;
  constexpr int GAE_CH = 4;
  const int rows_per = (T + GAE_CH - 1) / GAE_CH;
#pragma unroll
  for (int k = GAE_CH - 1; k >= 0; --k) {
    const int t0 = k * rows_per < T ? k * rows_per : T;
    const int t1 = t0 + rows_per < T ? t0 + rows_per : T;
    const int te = k == GAE_CH - 1 ? T + 1 : t1;       // the bootstrap row T travels with the last chunk
    for (int f = tid; f < (te - t0) * V4; f += 256) {
      const int t = t0 + f / V4, q = (f % V4) * 4;
      if (c0 + q < C) {
        const int64_t g = (int64_t)t * C + c0 + q;
        if (t < T) {
          cp_async16(&s_v[t * CW + q], value_preds + g);
          cp_async16(&s_w[t * CW + q], rewards + g);
        } else {
          cp_async16(&s_v[t * CW + q], use_gae ? next_value + c0 + q : value_preds + g);
        }
        cp_async16(&s_m[t * CW + q], masks + g);
        cp_async16(&s_b[t * CW + q], bad_masks + g);
      }
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
  }
  if (use_gae) {
    float g = 0.f;   // running GAE of this thread's column (threads < CW)
#pragma unroll
    for (int k = GAE_CH - 1; k >= 0; --k) {
      // chunks k-1 .. 0 may still be in flight
      if (k == 3) asm volatile("cp.async.wait_group 3;\n" ::: "memory");
      else if (k == 2) asm volatile("cp.async.wait_group 2;\n" ::: "memory");
      else if (k == 1) asm volatile("cp.async.wait_group 1;\n" ::: "memory");
      else asm volatile("cp.async.wait_group 0;\n" ::: "memory");
      __syncthreads();
      const int t0 = k * rows_per < T ? k * rows_per : T;
      const int t1 = t0 + rows_per < T ? t0 + rows_per : T;
      const int te = k == GAE_CH - 1 ? T + 1 : t1;
      if (k == GAE_CH - 1) {  // value_preds[-1] = next_value
        for (int f = tid; f < CW; f += 256)
          if (c0 + f < C) value_preds[(int64_t)T * C + c0 + f] = s_v[T * CW + f];
      }
      for (int f = t0 * CW + tid; f < te * CW; f += 256) s_v[f] = denorm(vc, s_v[f]);
      __syncthreads();
      for (int f = t0 * CW + tid; f < t1 * CW; f += 256) {
        float vn1 = s_v[f + CW], m1 = s_m[f + CW];
        // delta = r + gamma * V^[t+1] * m[t+1] - V^[t]
        s_w[f] = __fsub_rn(__fadd_rn(s_w[f], __fmul_rn(__fmul_rn(gamma, vn1), m1)), s_v[f]);
      }
      __syncthreads();
      if (tid < CW && c0 + tid < C) {
        // the recurrence is the critical path of the CTA: operands of 8 steps are pulled into registers first (their
        // addresses do not depend on g), so a step costs its three dependent roundings, not a shared-memory round trip
        for (int tb = t1 - 1; tb >= t0; tb -= 8) {
          float w[8], am[8], bb[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int t = tb - i;
            w[i] = am[i] = 0.f;
            bb[i] = 1.f;
            if (t >= t0) {
              w[i] = s_w[t * CW + tid];
              am[i] = __fmul_rn(gl, s_m[(t + 1) * CW + tid]);
              if (ptl) bb[i] = s_b[(t + 1) * CW + tid];
            }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int t = tb - i;
            if (t >= t0) {
              g = __fadd_rn(w[i], __fmul_rn(am[i], g));
              if (ptl) g = __fmul_rn(bb[i], g);
              s_w[t * CW + tid] = g;
            }
          }
        }
      }
      __syncthreads();
      for (int f = t0 * CW + tid; f < t1 * CW; f += 256) {
        int t = f / CW, c = f % CW;
        if (c0 + c < C) {
          float r = __fadd_rn(s_w[f], s_v[f]);
          returns[(int64_t)t * C + c0 + c] = r;
          if (adv) adv[(int64_t)t * C + c0 + c] = __fsub_rn(r, s_v[f]);
        }
      }
    }
  } else {
    cp_async_wait_all();
    __syncthreads();
    for (int f = tid; f < (T + 1) * CW; f += 256) s_v[f] = denorm(vc, s_v[f]);
    __syncthreads();
    // returns[-1] = next_value (raw); ret_t = (ret_{t+1}*gamma*m + r)*bad + (1-bad)*V^_t   (ptl)
    if (tid < CW && c0 + tid < C) {
      float ret = next_value[c0 + tid];
      returns[(int64_t)T * C + c0 + tid] = ret;
      for (int t = T - 1; t >= 0; --t) {
        float m1 = s_m[(t + 1) * CW + tid];
        float x = __fadd_rn(__fmul_rn(__fmul_rn(ret, gamma), m1), s_w[t * CW + tid]);
        if (ptl) {
          float b = s_b[(t + 1) * CW + tid];
          x = __fadd_rn(__fmul_rn(x, b), __fmul_rn(__fsub_rn(1.f, b), s_v[t * CW + tid]));
        }
        ret = x;
        s_w[t * CW + tid] = ret;
      }
    }
    __syncthreads();
    for (int f = tid; f < T * CW; f += 256) {
      int t = f / CW, c = f % CW;
      if (c0 + c < C) {
        float r = s_w[f];
        returns[(int64_t)t * C + c0 + c] = r;
        if (adv) adv[(int64_t)t * C + c0 + c] = __fsub_rn(r, s_v[f]);
      }
    }
  }
}

// ------------------------------------------------------------------ generic fallback: one thread per column
__global__ void gae_column_kernel(const float* __restrict__ rewards, float* __restrict__ value_preds,
                                  const float* __restrict__ masks, const float* __restrict__ bad_masks,
                                  const float* __restrict__ next_value, float* __restrict__ returns,
                                  float* __restrict__ adv, int T, int64_t C, float gamma, float gl, int use_gae, int ptl,
                                  const float* __restrict__ vn) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const VNConst vc = vn_load(vn);
  if (use_gae) {
    float nv = next_value[c];
    value_preds[(int64_t)T * C + c] = nv;
    float vnext = denorm(vc, nv), g = 0.f;
    for (int t = T - 1; t >= 0; --t) {
      int64_t i = (int64_t)t * C + c, i1 = i + C;
      float v = denorm(vc, value_preds[i]), m1 = masks[i1];
      float delta = __fsub_rn(__fadd_rn(rewards[i], __fmul_rn(__fmul_rn(gamma, vnext), m1)), v);
      g = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl, m1), g));
      if (ptl) g = __fmul_rn(bad_masks[i1], g);
      float r = __fadd_rn(g, v);
      returns[i] = r;
      if (adv) adv[i] = __fsub_rn(r, v);
      vnext = v;
    }
  } else {
    float ret = next_value[c];
    returns[(int64_t)T * C + c] = ret;
    for (int t = T - 1; t >= 0; --t) {
      int64_t i = (int64_t)t * C + c, i1 = i + C;
      float v = denorm(vc, value_preds[i]);
      float x = __fadd_rn(__fmul_rn(__fmul_rn(ret, gamma), masks[i1]), rewards[i]);
      if (ptl) {
        float b = bad_masks[i1];
        x = __fadd_rn(__fmul_rn(x, b), __fmul_rn(__fsub_rn(1.f, b), v));
      }
      ret = x;
      returns[i] = ret;
      if (adv) adv[i] = __fsub_rn(ret, v);
    }
  }
}

// ------------------------------------------------------------------ masked moments / normalisation
__global__ void __launch_bounds__(256) masked_moments_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                             int64_t n, double* __restrict__ out3) {
  double s = 0.0, q = 0.0, c = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    if (w == nullptr || w[i] != 0.f) { double v = (double)x[i]; s += v; q += v * v; c += 1.0; }
  }
  s = warp_sum_d(s); q = warp_sum_d(q); c = warp_sum_d(c);
  __shared__ double red[8][3];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { red[warp][0] = s; red[warp][1] = q; red[warp][2] = c; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
    atomicAdd(out3 + threadIdx.x, t);
  }
}

__global__ void normalize_kernel(const float* __restrict__ x, float* __restrict__ y, int64_t n,
                                 const double* __restrict__ m3) {
  const double cnt = m3[2];
  const double mean = m3[0] / cnt;
  double var = m3[1] / cnt - mean * mean;
  if (var < 0.0) var = 0.0;
  const float mf = (float)mean, df = __fadd_rn((float)sqrt(var), 1e-5f);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    y[i] = __fdiv_rn(__fsub_rn(x[i], mf), df);
}

// valuenorm.py:47-64
__global__ void valuenorm_update_kernel(float* vn, const double* __restrict__ m3, float beta, float omb) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    float bm = (float)(m3[0] / m3[2]), bsq = (float)(m3[1] / m3[2]);
    vn[0] = __fadd_rn(__fmul_rn(vn[0], beta), __fmul_rn(bm, omb));
    vn[1] = __fadd_rn(__fmul_rn(vn[1], beta), __fmul_rn(bsq, omb));
    vn[2] = __fadd_rn(__fmul_rn(vn[2], beta), omb);
  }
}

__global__ void valuenorm_apply_kernel(const float* __restrict__ vn, const float* __restrict__ x, float* __restrict__ y,
                                       int64_t n, int denormalize) {
  const VNConst c = vn_load(vn);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    y[i] = denormalize ? denorm(c, x[i]) : __fdiv_rn(__fsub_rn(x[i], c.mean), c.std);
}

static int stream_grid(int64_t n, int threads) {
  int64_t g = ceil_div64(n, threads);
  return (int)(g < 1 ? 1 : (g > 148 * 8 ? 148 * 8 : g));
}

}  // namespace hb

extern "C" {

int hb_gae_returns(const float* rewards, float* value_preds, const float* masks, const float* bad_masks,
                   const float* next_value, float* returns, float* advantages, int32_t T, int64_t C, float gamma,
                   float gamma_lambda, int use_gae, int use_proper_time_limits, const float* vn_state, void* stream) {
  using namespace hb;
  HB_CHECK_ARG(rewards && value_preds && masks && bad_masks && next_value && returns, "NULL buffer");
  HB_CHECK_ARG(T > 0 && C > 0, "T and C must be positive");
  cudaStream_t st = (cudaStream_t)stream;
  if (use_gae) {  // register-resident, time-segmented kernel (gae_seg.cu) for T <= 256
    int rc = HB_OK;
    if (hb::launch_gae_seg(rewards, value_preds, masks, bad_masks, next_value, returns, advantages, T, C, gamma, gamma_lambda,
                           use_proper_time_limits, vn_state, st, &rc))
      return rc;
  }
  const size_t per_col = (size_t)(4 * (size_t)T + 3) * sizeof(float);
  const size_t budget = 200 * 1024;
  int cw = 0;
  if (C % 4 == 0 && (((uintptr_t)rewards | (uintptr_t)value_preds | (uintptr_t)masks | (uintptr_t)bad_masks |
                      (uintptr_t)next_value) & 15) == 0) {
    // widest tile that fits shared memory while still giving >= 148 CTAs when the problem allows
    for (int w : {32, 16, 8, 4}) {
      if (per_col * w <= budget && (cw == 0 || ceil_div64(C, cw) < 148)) cw = w;
    }
  }
#define HB_GAE_TILED(W)                                                                                            \
  case W: {                                                                                                        \
    size_t smem = per_col * W;                                                                                     \
    cudaFuncSetAttribute(gae_tiled_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);             \
    gae_tiled_kernel<W><<<(unsigned)ceil_div64(C, W), 256, smem, st>>>(rewards, value_preds, masks, bad_masks,     \
                                                                      next_value, returns, advantages, T, C, gamma, \
                                                                      gamma_lambda, use_gae, use_proper_time_limits, \
                                                                      vn_state);                                   \
  } break;
  switch (cw) {
    HB_GAE_TILED(32) HB_GAE_TILED(16) HB_GAE_TILED(8) HB_GAE_TILED(4)
    default:
      gae_column_kernel<<<(unsigned)ceil_div64(C, 128), 128, 0, st>>>(rewards, value_preds, masks, bad_masks, next_value,
                                                                     returns, advantages, T, C, gamma, gamma_lambda,
                                                                     use_gae, use_proper_time_limits, vn_state);
  }
#undef HB_GAE_TILED
  HB_LAUNCH_DONE((cudaStream_t)stream,"hb_gae_returns");
  return HB_OK;
}

int hb_masked_moments(const float* x, const float* weight, int64_t n, double* out3, void* stream) {
  HB_CHECK_ARG(x && out3 && n >= 0, "bad argument");
  if (n == 0) return HB_OK;
  hb::masked_moments_kernel<<<hb::stream_grid(n, 256 * 4), 256, 0, (cudaStream_t)stream>>>(x, weight, n, out3);
  HB_LAUNCH_DONE((cudaStream_t)stream,"hb_masked_moments");
  return HB_OK;
}

int hb_normalize_by_moments(const float* x, float* x_out, int64_t n, const double* moments3, void* stream) {
  HB_CHECK_ARG(x && x_out && moments3 && n >= 0, "bad argument");
  if (n == 0) return HB_OK;
  hb::normalize_kernel<<<hb::stream_grid(n, 256 * 4), 256, 0, (cudaStream_t)stream>>>(x, x_out, n, moments3);
  HB_LAUNCH_DONE((cudaStream_t)stream,"hb_normalize_by_moments");
  return HB_OK;
}

int hb_valuenorm_update(float* vn_state, const double* moments3, double beta, void* stream) {
  HB_CHECK_ARG(vn_state && moments3, "NULL buffer");
  // the reference multiplies by the Python doubles beta and (1 - beta), each rounded to fp32 (valuenorm.py:62-64)
  hb::valuenorm_update_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(vn_state, moments3, (float)beta, (float)(1.0 - beta));
  HB_LAUNCH_DONE((cudaStream_t)stream,"hb_valuenorm_update");
  return HB_OK;
}

int hb_valuenorm_apply(const float* vn_state, const float* x, float* y, int64_t n, int denormalize, void* stream) {
  HB_CHECK_ARG(vn_state && x && y && n >= 0, "bad argument");
  if (n == 0) return HB_OK;
  hb::valuenorm_apply_kernel<<<hb::stream_grid(n, 256 * 4), 256, 0, (cudaStream_t)stream>>>(vn_state, x, y, n, denormalize);
  HB_LAUNCH_DONE((cudaStream_t)stream,"hb_valuenorm_apply");
  return HB_OK;
}
}
