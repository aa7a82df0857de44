// GAE scan, time-segmented and register-resident (sm_100a): the GAE branch of hb_gae_returns for T <= 256 (longer
// rollouts run the tiled kernel of gae.cu).
//
// Same arithmetic as gae_tiled_kernel (gae.cu), i.e. OnPolicyCriticBuffer{EP,FP}.compute_returns
// (harl/common/buffers/on_policy_critic_buffer_ep.py:97-140) + the advantage subtraction of
// harl/runners/on_policy_ha_runner.py:26-33 with every multiply / add separately rounded.
//
// Why another kernel: the [T+1, C] buffers of a C2 rollout are 19.7 MB -- 2.6 us of HBM time -- and the tiled kernel
// spends 13 us on them because only CW of its 256 threads walk the recurrence and every phase is fenced by a
// __syncthreads over shared memory.  Here a CTA is 32 columns x SEGS time segments, one warp per segment:
//   * every thread loads its own <= L steps of the four arrays straight from global into registers (128 B coalesced
//     per warp and row, ~100 independent loads per thread in flight at once, no staging pass, no shared-memory tile);
//   * delta_t and gamma*lambda*mask are formed in registers by all threads in parallel;
//   * the carry g between segments is the only cross-thread traffic (32 floats of shared memory per segment):
//       EXACT  : the warps run the recurrence in time order, later segment first, handing g over through a named
//                barrier (bar.arrive / bar.sync on 64 threads) -- bit-identical to the sequential reference; the
//                dependent chain is T steps of 2-3 roundings (~1.3 us at T = 200) but each warp stores its outputs
//                as soon as its own part is done, overlapped with the rest of the chain;
//       SCAN   : every warp first composes the affine map g_in -> g_out of its segment (A, B with FMAs), one
//                __syncthreads, then each thread folds the maps of the later segments (<= SEGS-1 FMAs) into its
//                incoming g and replays its own steps exactly.  The chain shrinks to 2L + SEGS steps; the carried g
//                differs from the sequential one by a few ulp (tests: <= 1e-6 of max|adv|), everything else is equal.
#include <stdlib.h>

#include "common.cuh"

namespace hb {

__device__ __forceinline__ void named_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void named_arrive(int id, int count) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

template <int SEGS, int L, bool PTL, bool SCAN>
__global__ void __launch_bounds__(32 * SEGS) gae_seg_kernel(const float* __restrict__ rewards, float* __restrict__ value_preds,
                                                            const float* __restrict__ masks, const float* __restrict__ bad_masks,
                                                            const float* __restrict__ next_value, float* __restrict__ returns,
                                                            float* __restrict__ adv, int T, int64_t C, float gamma, float gl,
                                                            const float* __restrict__ vn) {
  static_assert(SEGS <= 15, "one named barrier per hand-over");
  __shared__ float s_a[SEGS][32], s_b[SEGS][32];
  const int col = threadIdx.x & 31, seg = threadIdx.x >> 5;
  const int64_t c = (int64_t)blockIdx.x * 32 + col;
  const bool live = c < C;
  const int t0 = seg * L < T ? seg * L : T;
  const int t1 = t0 + L < T ? t0 + L : T;
  const int n = t1 - t0;              // steps of this segment (0 for segments past T)
  float w[L], am[L], vh[L], bb[PTL ? L : 1];
  float vlast = 0.f;                  // raw value at t1: the next segment's first row, or the bootstrap value
  if (live) {
    const int64_t base = (int64_t)t0 * C + c;
#pragma unroll
    for (int i = 0; i < L; ++i) {
      w[i] = am[i] = vh[i] = 0.f;
      if (PTL) bb[i] = 1.f;
      if (i < n) {
        const int64_t g = base + (int64_t)i * C;
        w[i] = __ldg(rewards + g);
        vh[i] = __ldg(value_preds + g);
        am[i] = __ldg(masks + g + C);
        if (PTL) bb[i] = __ldg(bad_masks + g + C);
      }
    }
    if (n > 0) vlast = t1 < T ? __ldg(value_preds + (int64_t)t1 * C + c) : __ldg(next_value + c);
    if (seg == 0) value_preds[(int64_t)T * C + c] = __ldg(next_value + c);   // value_preds[-1] = next_value (no thread reads row T)
  } else {
#pragma unroll
    for (int i = 0; i < L; ++i) {
      w[i] = am[i] = vh[i] = 0.f;
      if (PTL) bb[i] = 1.f;
    }
  }
  const VNConst vc = vn_load(vn);
  vlast = denorm(vc, vlast);
#pragma unroll
  for (int i = 0; i < L; ++i) vh[i] = denorm(vc, vh[i]);
#pragma unroll
  for (int i = 0; i < L; ++i) {
    // delta = r + gamma * V^[t+1] * m[t+1] - V^[t];   am = gamma*lambda * m[t+1]
    const float vnext = (i + 1 < L && i + 1 < n) ? vh[i + 1 < L ? i + 1 : 0] : vlast;
    w[i] = __fsub_rn(__fadd_rn(w[i], __fmul_rn(__fmul_rn(gamma, vnext), am[i])), vh[i]);
    am[i] = __fmul_rn(gl, am[i]);
  }
  float g = 0.f;
  if (SCAN) {
    float A = 1.f, B = 0.f;
#pragma unroll
    for (int i = L - 1; i >= 0; --i) {
      if (i < n) {
        float a = am[i], d = w[i];
        if (PTL) { a *= bb[i]; d *= bb[i]; }
        B = fmaf(a, B, d);
        A = a * A;
      }
    }
    s_a[seg][col] = A;
    s_b[seg][col] = B;
    __syncthreads();
    for (int k = SEGS - 1; k > seg; --k) g = fmaf(s_a[k][col], g, s_b[k][col]);
  } else {
    if (seg < SEGS - 1) {
      named_sync(seg + 1, 64);        // the later segment's carry is in s_a[seg + 1]
      g = s_a[seg + 1][col];
    }
  }
#pragma unroll
  for (int i = L - 1; i >= 0; --i) {
    if (i < n) {
      g = __fadd_rn(w[i], __fmul_rn(am[i], g));
      if (PTL) g = __fmul_rn(bb[i], g);
      w[i] = g;
    }
  }
  if (!SCAN && seg > 0) {
    s_a[seg][col] = g;
    __threadfence_block();
    named_arrive(seg, 64);
  }
  if (live) {
    const int64_t base = (int64_t)t0 * C + c;
#pragma unroll
    for (int i = 0; i < L; ++i) {
      if (i < n) {
        const float r = __fadd_rn(w[i], vh[i]);
        returns[base + (int64_t)i * C] = r;
        if (adv) adv[base + (int64_t)i * C] = __fsub_rn(r, vh[i]);
      }
    }
  }
}

// 1 = sequential carry (bit-exact), 2 = parallel-scan carry; -1: read HB_GAE_IMPL once (2, anything else gives 1)
static int g_gae_impl = -1;
int gae_impl() {
  if (g_gae_impl < 0) {
    const char* e = getenv("HB_GAE_IMPL");
    g_gae_impl = e != nullptr && atoi(e) == 2 ? 2 : 1;
  }
  return g_gae_impl;
}

template <int SEGS, int L>
static void launch_seg(bool ptl, bool scan, unsigned grid, cudaStream_t st, const float* rewards, float* value_preds,
                       const float* masks, const float* bad_masks, const float* next_value, float* returns, float* adv, int T,
                       int64_t C, float gamma, float gl, const float* vn) {
#define HB_SEG(P, S) gae_seg_kernel<SEGS, L, P, S><<<grid, 32 * SEGS, 0, st>>>(rewards, value_preds, masks, bad_masks, next_value, \
                                                                              returns, adv, T, C, gamma, gl, vn)
  if (ptl) { if (scan) HB_SEG(true, true); else HB_SEG(true, false); }
  else     { if (scan) HB_SEG(false, true); else HB_SEG(false, false); }
#undef HB_SEG
}

// Returns false if the shape is outside the kernel's range, T > 256 (the caller falls back to the tiled kernel).
bool launch_gae_seg(const float* rewards, float* value_preds, const float* masks, const float* bad_masks, const float* next_value,
                    float* returns, float* advantages, int T, int64_t C, float gamma, float gl, int ptl, const float* vn,
                    cudaStream_t st, int* rc) {
  if (T > 256) return false;
  const bool scan = gae_impl() == 2;
  const unsigned grid = (unsigned)ceil_div64(C, 32);
  // measured on B200 (profiles/gae_variants_r02.txt), T = 200: 13 segments x 16 steps wins for the sequential carry at
  // every width and for the scan below ~16k columns (shorter per-thread chains, 416 threads per CTA); 8 x 25 wins for
  // the scan on wide buffers (61 vs 84 us at 65536 columns: fewer, fatter threads keep more loads in flight per SM)
  const bool seg13 = T > 8 * 16 && T <= 13 * 16 && (!scan || C < 16384);
#define HB_GO(S, LL) launch_seg<S, LL>(ptl != 0, scan, grid, st, rewards, value_preds, masks, bad_masks, next_value, returns, \
                                       advantages, T, C, gamma, gl, vn)
  if (seg13) HB_GO(13, 16);
  else if (T <= 8 * 4) HB_GO(8, 4);
  else if (T <= 8 * 8) HB_GO(8, 8);
  else if (T <= 8 * 16) HB_GO(8, 16);
  else if (T <= 8 * 25) HB_GO(8, 25);
  else HB_GO(8, 32);
#undef HB_GO
  cudaError_t e = cudaGetLastError();
  *rc = e == cudaSuccess ? HB_OK : cuda_fail(e, "hb_gae_returns(seg)");
  if (e == cudaSuccess) note_launch("hb_gae_returns", st);
  return true;
}

}  // namespace hb

extern "C" {
int hb_set_gae_impl(int impl) {
  HB_CHECK_ARG(impl == 1 || impl == 2, "impl must be 1 (sequential carry) or 2 (parallel scan)");
  hb::g_gae_impl = impl;
  return HB_OK;
}
int hb_get_gae_impl(void) { return hb::gae_impl(); }
}
