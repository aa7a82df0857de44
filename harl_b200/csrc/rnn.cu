// GRU layer of the recurrent policies / critics (sm_100a): RNNLayer, harl/models/base/rnn.py:8-81.
//
// A recurrent batch is S steps x B sequences, rows step-major (row = s * B + j) -- the layout of the reference's
// sequence branch ([T*N, h] time-major, rnn.py:33-78) and of its chunk generators (Appendix D of SURVEY.md).
// The reference splits the sequence at reset steps and lets cuDNN/ATen run each segment; that is an optimisation
// of "h <- h * mask_t before every step" (verified bit-identical on CPU, SURVEY Appendix D), which is what runs here.
//
// Per layer: the input projection of ALL steps is one GEMM (gi = X W_ih^T + b_ih over S*B rows); the recurrence is
// S x (gh = hm W_hh^T + b_hh on B rows, then one elementwise gate kernel that also writes the masked state the next
// step multiplies).  Backward mirrors it: S x (gate backward, dhm += dgh W_hh), then the weight gradients and the
// input gradient as three GEMMs over all S*B rows.  The output LayerNorm is a row-wise kernel; its backward is
// fused into the head kernels (identity activation).  FP32 FFMA tiles (gemm_tile.cuh): the per-step GEMMs are
// [B, h] x [h, 3h] with h <= 256 -- latency-bound, not tensor-pipe work.
#include <math.h>
#include <stdlib.h>

#include <atomic>

#include "common.cuh"
#include "gemm_tile.cuh"
#include "kernels.cuh"
#include "rnn.cuh"
#include "row_helpers.cuh"

namespace hb {

// ------------------------------------------------------------------ Y (+)= X B + bias, any N (multiple of 4)
template <int NT, bool ACCUM>
__global__ void __launch_bounds__(256) linear_plain_kernel(const float* __restrict__ X, int ldx,
                                                           const float* __restrict__ Bm, int ldb,
                                                           const float* __restrict__ bias, float* __restrict__ Y, int ldy,
                                                           int64_t M, int N, int Kred) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GemmSmem<NT>& s = *reinterpret_cast<GemmSmem<NT>*>(smem_raw);
  constexpr int NCH = NT / 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t row0 = (int64_t)blockIdx.x * BM;
  const int n0 = blockIdx.y * NT;
  float acc[4][NT / 16];
  gemm_mainloop<NT, true>(X, ldx, Bm + n0, ldb, M, Kred, N - n0, row0, s, acc);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t row = row0 + ty * 4 + i;
    if (row >= M) continue;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int n = n0 + c * 64 + tx * 4;
      if (n >= N) continue;
      float4 o = make_float4(acc[i][c * 4 + 0], acc[i][c * 4 + 1], acc[i][c * 4 + 2], acc[i][c * 4 + 3]);
      if (bias != nullptr) {
        const float4 b = *reinterpret_cast<const float4*>(bias + n);
        o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
      }
      float4* dst = reinterpret_cast<float4*>(Y + row * ldy + n);
      if (ACCUM) { const float4 y = *dst; o.x += y.x; o.y += y.y; o.z += y.z; o.w += y.w; }
      *dst = o;
    }
  }
}

int launch_linear_plain(const float* X, int ldx, const float* Bm, int ldb, const float* bias, float* Y, int ldy,
                        int64_t M, int N, int Kred, bool accumulate, cudaStream_t st) {
  if (M <= 0) return HB_OK;
  constexpr int NT = 128;
  const size_t smem = sizeof(GemmSmem<NT>);
  dim3 grid((unsigned)ceil_div64(M, BM), (unsigned)((N + NT - 1) / NT));
  if (accumulate) linear_plain_kernel<NT, true><<<grid, 256, smem, st>>>(X, ldx, Bm, ldb, bias, Y, ldy, M, N, Kred);
  else linear_plain_kernel<NT, false><<<grid, 256, smem, st>>>(X, ldx, Bm, ldb, bias, Y, ldy, M, N, Kred);
  HB_LAUNCH_DONE(st, shape_label("rnn_linear", M, N, Kred));
  return HB_OK;
}

// ------------------------------------------------------------------ per-row mask gather + initial state
// mrow[r] = masks[src(r)];  hm0[j][:] = h0[src(j)][layer][:] * mrow[j]   (rnn.py:27-31, 60-70)
__global__ void rnn_mask_rows_kernel(const float* __restrict__ masks, const int32_t* __restrict__ index, int64_t M,
                                     float* __restrict__ mrow) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < M) mrow[r] = masks[index ? (int64_t)index[r] : r];
}

__global__ void rnn_init_state_kernel(const float* __restrict__ h0, const int32_t* __restrict__ index, int layer,
                                      int layers, int h, int64_t B, const float* __restrict__ mrow,
                                      float* __restrict__ hm0) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * h) return;
  const int64_t j = i / h;
  const int e = (int)(i % h);
  const int64_t src = index ? (int64_t)index[j] : j;
  hm0[i] = h0[(src * layers + layer) * h + e] * mrow[j];
}

// ------------------------------------------------------------------ gates, forward (PyTorch GRU, gate order r, z, n)
// r = s(gi_r + gh_r); z = s(gi_z + gh_z); n = tanh(gi_n + r * gh_n); h' = (1 - z) n + z hm
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

__global__ void gru_gate_fwd_kernel(const float* __restrict__ gi, const float* __restrict__ gh,
                                    const float* __restrict__ hm, int h, int64_t B, float* __restrict__ hs,
                                    float* __restrict__ gates, const float* __restrict__ mrow_next,
                                    float* __restrict__ hm_next, float* __restrict__ h_out, int out_stride) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * h) return;
  const int64_t b = i / h;
  const int e = (int)(i % h);
  const float* gir = gi + b * 3 * h;
  const float* ghr = gh + b * 3 * h;
  const float r = sigmoidf_(gir[e] + ghr[e]);
  const float z = sigmoidf_(gir[h + e] + ghr[h + e]);
  const float ghn = ghr[2 * h + e];
  const float n = tanhf(gir[2 * h + e] + r * ghn);
  const float hp = hm[i];
  const float hn = (1.f - z) * n + z * hp;
  hs[i] = hn;
  if (gates != nullptr) {
    float* g = gates + b * 4 * h;
    g[e] = r; g[h + e] = z; g[2 * h + e] = n; g[3 * h + e] = ghn;
  }
  if (hm_next != nullptr) hm_next[i] = hn * mrow_next[b];
  if (h_out != nullptr) h_out[b * out_stride + e] = hn;
}

// ------------------------------------------------------------------ gates, backward
// dh = dY_t + dhm_{t+1} * m_{t+1};  writes dgi_t, dgh_t and the direct part dh * z of d/d(hm_t)
__global__ void gru_gate_bwd_kernel(const float* __restrict__ dY, const float* __restrict__ dhm_next,
                                    const float* __restrict__ mrow_next, const float* __restrict__ gates,
                                    const float* __restrict__ hm, int h, int64_t B, float* __restrict__ dgi,
                                    float* __restrict__ dgh, float* __restrict__ dhm_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * h) return;
  const int64_t b = i / h;
  const int e = (int)(i % h);
  float dh = dY[i];
  if (dhm_next != nullptr) dh = fmaf(dhm_next[i], mrow_next[b], dh);
  const float* g = gates + b * 4 * h;
  const float r = g[e], z = g[h + e], n = g[2 * h + e], ghn = g[3 * h + e];
  const float hp = hm[i];
  const float dn_pre = dh * (1.f - z) * (1.f - n * n);
  const float dz_pre = dh * (hp - n) * z * (1.f - z);
  const float dr_pre = dn_pre * ghn * r * (1.f - r);
  float* a = dgi + b * 3 * h;
  float* c = dgh + b * 3 * h;
  a[e] = dr_pre; a[h + e] = dz_pre; a[2 * h + e] = dn_pre;
  c[e] = dr_pre; c[h + e] = dz_pre; c[2 * h + e] = dn_pre * r;
  dhm_out[i] = dh * z;
}

// ------------------------------------------------------------------ output LayerNorm (rnn.py:21,80), warp per row
__global__ void __launch_bounds__(ROW_THREADS) rnn_ln_fwd_kernel(const float* __restrict__ X, const float* __restrict__ lnw,
                                                                 const float* __restrict__ lnb, float* __restrict__ Y,
                                                                 float* __restrict__ stats, int64_t rows, int N) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = (int64_t)blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), nw = (int64_t)gridDim.x * ROW_WARPS;
  const float inv_n = 1.f / (float)N;
  for (int64_t r = w0; r < rows; r += nw) {
    float v[8];
    float s = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) { int n = lane + 32 * q; v[q] = n < N ? X[r * N + n] : 0.f; s += v[q]; }
    const float mean = warp_sum(s) * inv_n;
    float sq = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) { int n = lane + 32 * q; if (n < N) { float dlt = v[q] - mean; sq = fmaf(dlt, dlt, sq); } }
    const float rstd = rsqrtf(warp_sum(sq) * inv_n + 1e-5f);
#pragma unroll
    for (int q = 0; q < 8; ++q) { int n = lane + 32 * q; if (n < N) Y[r * N + n] = (v[q] - mean) * rstd * lnw[n] + lnb[n]; }
    if (stats != nullptr && lane == 0) { stats[r * 2] = mean; stats[r * 2 + 1] = rstd; }
  }
}

// ------------------------------------------------------------------ persistent per-sequence recurrence (default)
// hb_set_rnn_impl(1), the default, for h = 64 (other widths run the per-step kernels).  One warp owns one sequence for all S steps: W_hh^T (64 x 192
// floats, regrouped so that lane l finds the r, z, n weights of its two hidden units 2l, 2l+1 in two LDS.128 per input
// unit) stays in shared memory, the state stays in registers (unit i lives in lane i/2, broadcast by shuffle), and per
// step the warp reads its gi row and the reset mask and writes hm / hs / gates exactly as the per-step kernels do.
// Accumulation order matches the tiled GEMM (ascending input unit from zero, bias added last), so the results are
// bit-identical to the launch-per-step path (tests/test_gpu_rnn.py).  Replaces 2 S launches per layer by one.
constexpr int GP_H = 64;
__global__ void __launch_bounds__(256) gru_seq_fwd_kernel(const float* __restrict__ whh_t /* [64][192] */,
                                                          const float* __restrict__ bhh /* [192] */,
                                                          const float* __restrict__ gi /* [S*B, 192] */,
                                                          const float* __restrict__ h0, const int32_t* __restrict__ index,
                                                          int layer, int layers, const float* __restrict__ mrow,
                                                          int64_t S, int64_t B, float* __restrict__ hm,
                                                          float* __restrict__ hs, float* __restrict__ gates,
                                                          float* __restrict__ h_out) {
  // [64 input units][2 parts][32 lanes][4]: part 0 = {r0, r1, z0, z1}, part 1 = {n0, n1, -, -} of lane l's units 2l, 2l+1
  // (consecutive lanes read consecutive float4: conflict-free LDS.128)
  extern __shared__ __align__(16) float gp_w[];
  for (int f = threadIdx.x; f < GP_H * 2 * 32 * 4; f += 256) {
    const int i = f >> 8, part = (f >> 7) & 1, l = (f >> 2) & 31, c = part * 4 + (f & 3);
    gp_w[f] = c < 6 ? whh_t[i * 3 * GP_H + (c >> 1) * GP_H + 2 * l + (c & 1)] : 0.f;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int e = 2 * lane;
  const float2 br = *reinterpret_cast<const float2*>(bhh + e), bz = *reinterpret_cast<const float2*>(bhh + GP_H + e),
               bn = *reinterpret_cast<const float2*>(bhh + 2 * GP_H + e);
  for (int64_t j = (int64_t)blockIdx.x * 8 + warp; j < B; j += (int64_t)gridDim.x * 8) {
    const int64_t src = index ? (int64_t)index[j] : j;
    float2 h = *reinterpret_cast<const float2*>(h0 + (src * layers + layer) * GP_H + e);
    for (int64_t t = 0; t < S; ++t) {
      const int64_t row = t * B + j;
      const float m = mrow[row];
      const float hm0 = h.x * m, hm1 = h.y * m;
      *reinterpret_cast<float2*>(hm + row * GP_H + e) = make_float2(hm0, hm1);
      float a[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
      for (int ii = 0; ii < 32; ++ii) {
        const float v0 = __shfl_sync(0xffffffffu, hm0, ii), v1 = __shfl_sync(0xffffffffu, hm1, ii);
        const float4* w0 = reinterpret_cast<const float4*>(gp_w + ((2 * ii) * 64 + lane) * 4);      // unit 2 ii
        const float4* w1 = reinterpret_cast<const float4*>(gp_w + ((2 * ii + 1) * 64 + lane) * 4);  // unit 2 ii + 1
        const float4 p = w0[0], q = w0[32];
        a[0] = fmaf(v0, p.x, a[0]); a[1] = fmaf(v0, p.y, a[1]); a[2] = fmaf(v0, p.z, a[2]);
        a[3] = fmaf(v0, p.w, a[3]); a[4] = fmaf(v0, q.x, a[4]); a[5] = fmaf(v0, q.y, a[5]);
        const float4 p1 = w1[0], q1 = w1[32];
        a[0] = fmaf(v1, p1.x, a[0]); a[1] = fmaf(v1, p1.y, a[1]); a[2] = fmaf(v1, p1.z, a[2]);
        a[3] = fmaf(v1, p1.w, a[3]); a[4] = fmaf(v1, q1.x, a[4]); a[5] = fmaf(v1, q1.y, a[5]);
      }
      const float* g = gi + row * 3 * GP_H;
      const float2 gr = *reinterpret_cast<const float2*>(g + e), gz = *reinterpret_cast<const float2*>(g + GP_H + e),
                   gn = *reinterpret_cast<const float2*>(g + 2 * GP_H + e);
      const float ghr0 = a[0] + br.x, ghr1 = a[1] + br.y, ghz0 = a[2] + bz.x, ghz1 = a[3] + bz.y;
      const float ghn0 = a[4] + bn.x, ghn1 = a[5] + bn.y;
      const float r0 = sigmoidf_(gr.x + ghr0), r1 = sigmoidf_(gr.y + ghr1);
      const float z0 = sigmoidf_(gz.x + ghz0), z1 = sigmoidf_(gz.y + ghz1);
      const float n0 = tanhf(gn.x + r0 * ghn0), n1 = tanhf(gn.y + r1 * ghn1);
      h.x = (1.f - z0) * n0 + z0 * hm0;
      h.y = (1.f - z1) * n1 + z1 * hm1;
      *reinterpret_cast<float2*>(hs + row * GP_H + e) = h;
      if (gates != nullptr) {
        float* gt = gates + row * 4 * GP_H;
        *reinterpret_cast<float2*>(gt + e) = make_float2(r0, r1);
        *reinterpret_cast<float2*>(gt + GP_H + e) = make_float2(z0, z1);
        *reinterpret_cast<float2*>(gt + 2 * GP_H + e) = make_float2(n0, n1);
        *reinterpret_cast<float2*>(gt + 3 * GP_H + e) = make_float2(ghn0, ghn1);
      }
    }
    if (h_out != nullptr) *reinterpret_cast<float2*>(h_out + (j * layers + layer) * GP_H + e) = h;
  }
}

// -1: read HB_RNN_IMPL once; 0 = launch per step ("per_step"), 1 = persistent per-sequence kernel (default since round 2:
// GPU-verified bit-for-bit against the per-step kernels, tests/test_gpu_rnn.py; h = 64 only, other widths run per step)
static std::atomic<int> g_rnn_impl{-1};
int rnn_impl() {
  int v = g_rnn_impl.load(std::memory_order_relaxed);
  if (v < 0) {
    const char* e = getenv("HB_RNN_IMPL");
    v = (e != nullptr && strcmp(e, "per_step") == 0) ? 0 : 1;
    g_rnn_impl.store(v);
  }
  return v;
}
void set_rnn_impl(int v) { g_rnn_impl.store(v ? 1 : 0); }

// ------------------------------------------------------------------ workspace
size_t rnn_work_floats(const PrepLayout& Q, int64_t M, int grad) {
  if (!Q.rnn_layers) return 0;
  const size_t h = Q.rh, m = (size_t)M, R = Q.rnn_layers;
  size_t f = (m + 3) / 4 * 4;                                           // mrow
  f += R * (m * 3 * h + m * h + m * h);                                 // gi, hm, hs per layer
  f += m * 3 * h;                                                       // gh scratch (B <= M rows)
  f += m * h + (size_t)round_up((int)(2 * M), 4);                       // out, stats
  if (grad) f += R * m * 4 * h + 2 * m * 3 * h + 2 * m * h + 3 * m * h; // gates; dgi, dgh; dhm x2; dtop, dxA, dxB
  return f;
}

int carve_rnn(const PrepLayout& Q, int64_t M, int grad, float* p, RnnWork* w) {
  memset(w, 0, sizeof(*w));
  if (!Q.rnn_layers) return HB_OK;
  const size_t h = Q.rh, m = (size_t)M;
  w->mrow = p; p += round_up((int)M, 4);
  for (int l = 0; l < Q.rnn_layers; ++l) {
    w->gi[l] = p; p += m * 3 * h;
    w->hm[l] = p; p += m * h;
    w->hs[l] = p; p += m * h;
  }
  w->gh = p; p += m * 3 * h;
  w->out = p; p += m * h;
  w->stats = p; p += round_up((int)(2 * M), 4);
  if (grad) {
    for (int l = 0; l < Q.rnn_layers; ++l) { w->gates[l] = p; p += m * 4 * h; }
    w->dgi = p; p += m * 3 * h;
    w->dgh = p; p += m * 3 * h;
    w->dhm[0] = p; p += m * h;
    w->dhm[1] = p; p += m * h;
    w->dtop = p; p += m * h;
    w->dx[0] = p; p += m * h;
    w->dx[1] = p; p += m * h;
  }
  return HB_OK;
}

static inline unsigned ew_grid(int64_t n) { return (unsigned)ceil_div64(n, 256); }

// ------------------------------------------------------------------ forward over S steps x B sequences
int rnn_forward(const PrepLayout& Q, const float* prep, const float* X, int64_t S, int64_t B, const float* h0,
                const float* masks, const int32_t* index, float* h_out, const RnnWork& w, cudaStream_t st) {
  const int h = Q.rh, R = Q.rnn_layers;
  const int64_t M = S * B;
  rnn_mask_rows_kernel<<<ew_grid(M), 256, 0, st>>>(masks, index, M, w.mrow);
  HB_LAUNCH_DONE(st, "rnn_mask_rows");
  const float* xin = X;
  int rc;
  for (int l = 0; l < R; ++l) {
    if ((rc = launch_linear_plain(xin, h, prep + Q.rnn_wih_t[l], 3 * h, prep + Q.rnn_bih[l], w.gi[l], 3 * h, M, 3 * h, h,
                                  false, st)))
      return rc;
    if (rnn_impl() == 1 && h == GP_H) {  // persistent recurrence (see gru_seq_fwd_kernel)
      const size_t smem = (size_t)GP_H * 32 * 8 * sizeof(float);
      static bool attr_done = false;
      if (!attr_done) {
        cudaFuncSetAttribute(gru_seq_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        attr_done = true;
      }
      int64_t g = ceil_div64(B, 8);
      if (g > 148 * 3) g = 148 * 3;
      gru_seq_fwd_kernel<<<(unsigned)g, 256, smem, st>>>(prep + Q.rnn_whh_t[l], prep + Q.rnn_bhh[l], w.gi[l], h0, index, l, R,
                                                        w.mrow, S, B, w.hm[l], w.hs[l], w.gates[l], h_out);
      HB_LAUNCH_DONE(st, shape_label("rnn_gru_seq_fwd", S * B, h, (int)S));
      xin = w.hs[l];
      continue;
    }
    rnn_init_state_kernel<<<ew_grid(B * h), 256, 0, st>>>(h0, index, l, R, h, B, w.mrow, w.hm[l]);
    HB_LAUNCH_DONE(st, "rnn_init_state");
    for (int64_t t = 0; t < S; ++t) {
      const float* hm_t = w.hm[l] + t * B * h;
      if ((rc = launch_linear_plain(hm_t, h, prep + Q.rnn_whh_t[l], 3 * h, prep + Q.rnn_bhh[l], w.gh, 3 * h, B, 3 * h, h,
                                    false, st)))
        return rc;
      const bool last = t + 1 == S;
      gru_gate_fwd_kernel<<<ew_grid(B * h), 256, 0, st>>>(
          w.gi[l] + t * B * 3 * h, w.gh, hm_t, h, B, w.hs[l] + t * B * h,
          w.gates[l] ? w.gates[l] + t * B * 4 * h : nullptr, last ? nullptr : w.mrow + (t + 1) * B,
          last ? nullptr : w.hm[l] + (t + 1) * B * h, (last && h_out) ? h_out + (int64_t)l * h : nullptr, R * h);
      HB_LAUNCH_DONE(st, "rnn_gru_gate_fwd");
    }
    xin = w.hs[l];
  }
  rnn_ln_fwd_kernel<<<row_grid(M), ROW_THREADS, 0, st>>>(w.hs[R - 1], prep + Q.rnn_lnw, prep + Q.rnn_lnb, w.out, w.stats, M, h);
  HB_LAUNCH_DONE(st, shape_label("rnn_ln_fwd", M, h, 0));
  return HB_OK;
}

// ------------------------------------------------------------------ backward (BPTT) given w.dtop = d loss / d hs[R-1]
// X: the layer-0 input sequence (trunk output).  Writes d loss / d X to *dX_out (one of w.dx[]).
int rnn_backward(const ParamLayout& P, const PrepLayout& Q, const float* params, const float* X, int64_t S, int64_t B,
                 float* grad, const RnnWork& w, float** dX_out, cudaStream_t st) {
  const int h = Q.rh, R = Q.rnn_layers;
  const int64_t M = S * B;
  const float* dY = w.dtop;
  int rc;
  for (int l = R - 1; l >= 0; --l) {
    int cur = 0;
    for (int64_t t = S - 1; t >= 0; --t) {
      const bool last = t + 1 == S;
      float* dhm_t = w.dhm[cur ^ 1];
      gru_gate_bwd_kernel<<<ew_grid(B * h), 256, 0, st>>>(
          dY + t * B * h, last ? nullptr : w.dhm[cur], last ? nullptr : w.mrow + (t + 1) * B,
          w.gates[l] + t * B * 4 * h, w.hm[l] + t * B * h, h, B, w.dgi + t * B * 3 * h, w.dgh + t * B * 3 * h, dhm_t);
      HB_LAUNCH_DONE(st, "rnn_gru_gate_bwd");
      // d/d(hm_t) += dgh_t W_hh   (W_hh [3h][h] as stored)
      if (t > 0) {
        if ((rc = launch_linear_plain(w.dgh + t * B * 3 * h, 3 * h, params + P.rnn_whh[l], h, nullptr, dhm_t, h, B, h,
                                      3 * h, true, st)))
          return rc;
      }
      cur ^= 1;
    }
    const float* xin = l == 0 ? X : w.hs[l - 1];
    if ((rc = launch_dw_accum(w.dgh, 3 * h, w.hm[l], h, h, grad + P.rnn_whh[l], grad + P.rnn_bhh[l], M, st))) return rc;
    if ((rc = launch_dw_accum(w.dgi, 3 * h, xin, h, h, grad + P.rnn_wih[l], grad + P.rnn_bih[l], M, st))) return rc;
    float* dx = w.dx[l & 1];
    if ((rc = launch_linear_plain(w.dgi, 3 * h, params + P.rnn_wih[l], h, nullptr, dx, h, M, h, 3 * h, false, st))) return rc;
    dY = dx;
    *dX_out = dx;
  }
  return HB_OK;
}

// ------------------------------------------------------------------ tangent (forward-mode) pass, trust-region FVP
// gate tangents from the saved gates (r, z, n, ghn), the tangents of the two projections and of the masked state:
//   rd = r(1-r)(gid_r + ghd_r);  zd = z(1-z)(gid_z + ghd_z);  nd = (1-n^2)(gid_n + rd ghn + r ghd_n)
//   hd = (1-z) nd + zd (hm - n) + z hmd
__global__ void gru_gate_jvp_kernel(const float* __restrict__ gid, const float* __restrict__ ghd,
                                    const float* __restrict__ gates, const float* __restrict__ hm,
                                    const float* __restrict__ hmd, int h, int64_t B, float* __restrict__ hsd,
                                    const float* __restrict__ mrow_next, float* __restrict__ hmd_next) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * h) return;
  const int64_t b = i / h;
  const int e = (int)(i % h);
  const float* a = gid + b * 3 * h;
  const float* c = ghd + b * 3 * h;
  const float* g = gates + b * 4 * h;
  const float r = g[e], z = g[h + e], n = g[2 * h + e], ghn = g[3 * h + e];
  const float rd = r * (1.f - r) * (a[e] + c[e]);
  const float zd = z * (1.f - z) * (a[h + e] + c[h + e]);
  const float nd = (1.f - n * n) * (a[2 * h + e] + rd * ghn + r * c[2 * h + e]);
  const float hd = (1.f - z) * nd + zd * (hm[i] - n) + z * (hmd != nullptr ? hmd[i] : 0.f);
  hsd[i] = hd;
  if (hmd_next != nullptr) hmd_next[i] = hd * mrow_next[b];
}

// tangent of the output LayerNorm: yd = gd xh + bd + g rstd (hd - mean(hd) - xh mean(xh hd)), xh = (hs - mu) rstd
__global__ void __launch_bounds__(ROW_THREADS) rnn_ln_jvp_kernel(const float* __restrict__ X, const float* __restrict__ Xd,
                                                                 const float* __restrict__ stats,
                                                                 const float* __restrict__ lnw, const float* __restrict__ lnwd,
                                                                 const float* __restrict__ lnbd, float* __restrict__ Yd,
                                                                 int64_t rows, int N) {
  const int lane = threadIdx.x & 31;
  const int64_t w0 = (int64_t)blockIdx.x * ROW_WARPS + (threadIdx.x >> 5), nw = (int64_t)gridDim.x * ROW_WARPS;
  const float inv_n = 1.f / (float)N;
  for (int64_t r = w0; r < rows; r += nw) {
    const float mu = stats[r * 2], rstd = stats[r * 2 + 1];
    float xh[8], xd[8];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      int n = lane + 32 * q;
      xh[q] = xd[q] = 0.f;
      if (n < N) { xh[q] = (X[r * N + n] - mu) * rstd; xd[q] = Xd[r * N + n]; s1 += xd[q]; s2 = fmaf(xd[q], xh[q], s2); }
    }
    const float m1 = warp_sum(s1) * inv_n, m2 = warp_sum(s2) * inv_n;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      int n = lane + 32 * q;
      if (n < N) Yd[r * N + n] = lnwd[n] * xh[q] + lnbd[n] + lnw[n] * rstd * (xd[q] - m1 - xh[q] * m2);
    }
  }
}

size_t rnn_jvp_floats(const PrepLayout& Q, int64_t M) {
  if (!Q.rnn_layers) return 0;
  const size_t h = Q.rh, m = (size_t)M;
  return m * 3 * h + m * 3 * h + (size_t)Q.rnn_layers * 2 * m * h + m * h;  // gid, ghd, (hmd, hsd) per layer, outd
}

int carve_rnn_jvp(const PrepLayout& Q, int64_t M, float* p, RnnJvpWork* w) {
  memset(w, 0, sizeof(*w));
  if (!Q.rnn_layers) return HB_OK;
  const size_t h = Q.rh, m = (size_t)M;
  w->gid = p; p += m * 3 * h;
  w->ghd = p; p += m * 3 * h;
  for (int l = 0; l < Q.rnn_layers; ++l) { w->hmd[l] = p; p += m * h; w->hsd[l] = p; p += m * h; }
  w->outd = p;
  return HB_OK;
}

// Xd: tangent of the layer-0 input sequence; tprep: tangent of the prepared weights (trpo.cu tangent_prepare).
// Needs the forward pass of the SAME batch in w (gradient mode: gates saved).  Result: jw.outd = tangent of w.out.
int rnn_jvp_forward(const PrepLayout& Q, const float* prep, const float* tprep, const float* X, const float* Xd, int64_t S,
                    int64_t B, const RnnWork& w, const RnnJvpWork& jw, cudaStream_t st) {
  const int h = Q.rh, R = Q.rnn_layers;
  const int64_t M = S * B;
  const float* xin = X;
  const float* xd = Xd;
  int rc;
  for (int l = 0; l < R; ++l) {
    // gid = Xd W_ih^T + X Wd_ih^T + bd_ih over all steps
    if ((rc = launch_linear_plain(xd, h, prep + Q.rnn_wih_t[l], 3 * h, tprep + Q.rnn_bih[l], jw.gid, 3 * h, M, 3 * h, h, false, st))) return rc;
    if ((rc = launch_linear_plain(xin, h, tprep + Q.rnn_wih_t[l], 3 * h, nullptr, jw.gid, 3 * h, M, 3 * h, h, true, st))) return rc;
    for (int64_t t = 0; t < S; ++t) {
      const float* hm_t = w.hm[l] + t * B * h;
      const float* hmd_t = t == 0 ? nullptr : jw.hmd[l] + t * B * h;  // the stored initial state carries no tangent
      // ghd = hmd W_hh^T + hm Wd_hh^T + bd_hh
      if ((rc = launch_linear_plain(hm_t, h, tprep + Q.rnn_whh_t[l], 3 * h, tprep + Q.rnn_bhh[l], jw.ghd, 3 * h, B, 3 * h, h, false, st))) return rc;
      if (hmd_t != nullptr &&
          (rc = launch_linear_plain(hmd_t, h, prep + Q.rnn_whh_t[l], 3 * h, nullptr, jw.ghd, 3 * h, B, 3 * h, h, true, st)))
        return rc;
      const bool last = t + 1 == S;
      gru_gate_jvp_kernel<<<ew_grid(B * h), 256, 0, st>>>(jw.gid + t * B * 3 * h, jw.ghd, w.gates[l] + t * B * 4 * h, hm_t,
                                                         hmd_t, h, B, jw.hsd[l] + t * B * h,
                                                         last ? nullptr : w.mrow + (t + 1) * B,
                                                         last ? nullptr : jw.hmd[l] + (t + 1) * B * h);
      HB_LAUNCH_DONE(st, "rnn_gru_gate_jvp");
    }
    xin = w.hs[l];
    xd = jw.hsd[l];
  }
  rnn_ln_jvp_kernel<<<row_grid(M), ROW_THREADS, 0, st>>>(w.hs[R - 1], xd, w.stats, prep + Q.rnn_lnw, tprep + Q.rnn_lnw,
                                                        tprep + Q.rnn_lnb, jw.outd, M, h);
  HB_LAUNCH_DONE(st, shape_label("rnn_ln_jvp", M, h, 0));
  return HB_OK;
}

}  // namespace hb
