// Fused actor / critic update kernel (SURVEY.md section 7 step 4, section 8(d) "fused actor update"):
//   ONE persistent launch per (agent, epoch, minibatch) does, per 128-row tile, entirely on chip,
//     obs rows -> feature LayerNorm -> [Linear -> act -> LayerNorm] x 2 -> head -> PPO-clip / value loss
//     -> d logits -> head backward -> LayerNorm/act backward x 2 -> weight-gradient accumulation,
//   so per row and epoch the kernel reads the algorithmic bytes only (obs + a handful of scalars) and no activation ever
//   touches HBM.  Replaces HAPPO.update's forward / loss / backward (harl/algorithms/actors/happo.py:28-91 over
//   harl/models/base/mlp.py:25-36, act.py, distributions.py) and VCritic.update's (v_critic.py:75-146).
//
// Arithmetic: every GEMM runs on tcgen05 (kind::f16, fp32 accumulators in TMEM) with the error-compensated split
//   x = hi + lo (hi = fp16(x), lo = fp16(x - hi), operands pre-scaled by powers of two into the fp16 range):
//   D += A_hi B_hi + A_lo B_hi + A_hi B_lo -- 22-bit operands, the accuracy class of the 3xTF32 path (measured on a B200:
//   profiles/probe_umma_layouts_r02.log) at twice its MMA rate and half its shared-memory footprint.
//
// LayerNorm affines are folded into the NEXT layer's weights (W' = W diag(gamma), b' = b + W beta; hb_net_prepare packs
// the images), so the on-chip activations are the plain normalised rows xhat, the LayerNorm backward needs no per-row
// affine work, and all affine gradients fall out of the weight gradients afterwards (optim.cu featnorm_grad_fold_kernel,
// applied per layer).
//
// Layout trick: a tile image written by "thread = row" as  IMG[row/8][feature/8][row%8][8 x fp16]  is at the same time a
//   K-major operand (rows x features: the forward / dX GEMMs) and an MN-major operand (features x rows: the weight-gradient
//   GEMMs, whose reduction index is the row) -- no transposition anywhere (umma.cuh).  dZ overwrites xhat in place.
//
// CTA = 6 warps: warp 0 streams weight chunks through a TMA ring, warp 1 issues the MMAs, warps 2-5 (thread = row, TMEM
// lane quarter = warp % 4) run the epilogues.  The phases of a tile alternate strictly between the MMA warp and the
// epilogue warps (two mbarriers); weight gradients accumulate in TMEM across all tiles of the CTA and are written once,
// to the CTA's slot of a split buffer (deterministic; summed by fused_slot_reduce_kernel).
#include <cuda_fp16.h>

#include <atomic>

#include "common.cuh"
#include "head_rows.cuh"
#include "kernels.cuh"
#include "row_helpers.cuh"
#include "fused_args.cuh"
#include "umma.cuh"

namespace hb {

int launch_featnorm_fold_at(const float* params, float* grad, int w0, int b0, int gw, int gb, int N, int K, cudaStream_t st);

namespace fz {

constexpr float XS = 16.f;          // activation images hold XS * xhat      (|xhat| <= sqrt(h))
constexpr float DZS = 16.f;         // gradient images hold DZS * dZ (dZ is un-normalised: O(advantage))
constexpr int TILE = 128;
constexpr int NH = 16;              // padded head width (MMA N)
constexpr int MAX_STAGES = 3;          // weight-chunk ring: 3 stages when the images leave room (in_dim <= 32), else 2
constexpr int STAGE_BYTES = 16384;  // one weight chunk: hi + lo images of [128][32] fp16
constexpr int THREADS = 320;           // producer warp, MMA warp, 8 epilogue warps (two threads per row)
enum { M_GRAD = 0, M_EVAL = 1 };

// TMEM columns (fp32 accumulators, 128 lanes each)
constexpr uint32_t C_F = 0;         // forward pre-activations / backward dY      [rows][<= 128]
constexpr uint32_t C_W1 = 128;      // dW'_1                                       [n][k <= 128]
constexpr uint32_t C_W0 = 256;      // dW'_0                                       [n][k <= 64]
constexpr uint32_t C_H = 320;       // head outputs                                [rows][16]
constexpr uint32_t C_WH = 336;      // dW'_head transposed                         [feature][16]
constexpr uint32_t C_B1 = 352;      // db'_1 in column 0                           [n][16]
constexpr uint32_t C_B0 = 368;      // db'_0 in column 0
constexpr uint32_t C_BH = 384;      // column sums of the d-logits image: lane j = db'_head[j]; Box: lane 8 + j = d log_std[j]
constexpr uint32_t TMEM_COLS = 512;



// ------------------------------------------------------------------------------------------------ image addressing
// byte offset of (row r, 8-feature chunk ch) in a tile image with `wch` chunks per row
__device__ __forceinline__ uint32_t img_off(int r, int ch, int wch) { return (uint32_t)(((r >> 3) * wch + ch) * 128 + (r & 7) * 16); }

struct Op {  // one operand view for the MMA issuer
  uint32_t hi, lo, lbo, sbo, adv;
};
__device__ __forceinline__ Op op_kmajor(uint32_t base, uint32_t img_bytes, int wch, int ch0) {  // rows x features, k offset = chunk ch0
  return Op{base + (uint32_t)ch0 * 128u, base + img_bytes + (uint32_t)ch0 * 128u, 128u, (uint32_t)wch * 128u, 256u};
}
__device__ __forceinline__ Op op_mnmajor(uint32_t base, uint32_t img_bytes, int wch, int ch0) {  // features x rows, feature offset = chunk ch0
  return Op{base + (uint32_t)ch0 * 128u, base + img_bytes + (uint32_t)ch0 * 128u, (uint32_t)wch * 128u, 128u, 2u * (uint32_t)wch * 128u};
}
// D (+)= A B^T over `ksteps` MMA k-steps, three passes per step (b_lo == 0: B is exact in fp16 -> two passes)
__device__ __forceinline__ void gemm3(uint32_t d, const Op& A, const Op& B, int ksteps, uint32_t idesc, bool accumulate, bool b_has_lo = true) {
  for (int ks = 0; ks < ksteps; ++ks) {
    const uint64_t ah = um::desc(A.hi + ks * A.adv, A.lbo, A.sbo), al = um::desc(A.lo + ks * A.adv, A.lbo, A.sbo);
    const uint64_t bh = um::desc(B.hi + ks * B.adv, B.lbo, B.sbo);
    um::mma_f16(d, ah, bh, idesc, (accumulate || ks > 0) ? 1u : 0u);
    um::mma_f16(d, al, bh, idesc, 1u);
    if (b_has_lo) {
      const uint64_t bl = um::desc(B.lo + ks * B.adv, B.lbo, B.sbo);
      um::mma_f16(d, ah, bl, idesc, 1u);
    }
  }
}

// ------------------------------------------------------------------------------------------------ epilogue pieces
// d act / dz from the post-activation value and the sign of z
template <int ACT>
__device__ __forceinline__ float act_prime(int act_rt, float a, bool zpos) {
  const int A_ = ACT >= 0 ? ACT : act_rt;
  switch (A_) {
    case HB_ACT_RELU: return zpos ? 1.f : 0.f;
    case HB_ACT_TANH: return 1.f - a * a;
    case HB_ACT_SIGMOID: return a * (1.f - a);
    case HB_ACT_LEAKY_RELU: return zpos ? 1.f : 0.01f;
    case HB_ACT_SELU: {
      const float al = 1.6732632423543772848170429916717f, s = 1.0507009873554804934193349852946f;
      return zpos ? s : a + s * al;   // s * al * exp(z) = a + s * al for z <= 0
    }
    default: return 1.f;
  }
}
template <int ACT>
__device__ __forceinline__ float act_f(int act_rt, float z) {
  if (ACT >= 0) return act_fwd<(ACT >= 0 ? ACT : 0)>(z);
  return act_fwd_rt(act_rt, z);
}

// Two threads share a row (column halves): partial row sums meet through shared memory and a 64-thread named barrier of
// the two warps that own the same TMEM lane quarter.  Both threads form a + b in the same order (bit-identical results).
struct RowPair {
  float* xch;     // [2 halves][128 rows][2 slots]
  int half, r, bar_id;
  __device__ __forceinline__ void put(int slot, float v) const { xch[(half * TILE + r) * 2 + slot] = v; }
  __device__ __forceinline__ void sync() const { asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory"); }
  __device__ __forceinline__ float total(int slot, float mine) const {
    const float other = xch[((half ^ 1) * TILE + r) * 2 + slot];
    return half == 0 ? mine + other : other + mine;
  }
};

// ---- single-pass epilogues.  TMEM reads are the scarce resource here (measured: ~64 B / cycle / SM, so every extra pass over
// a 128 x 128 accumulator costs ~1000 cycles per tile): each accumulator element is read ONCE, the thread's <= 64 columns stay
// in registers for the statistics and the write-back.  The next 16-column chunk's tcgen05.ld is in flight while the current
// one is consumed (two alternating register buffers; the loops are fully unrolled so that every index is static).

// Linear -> act -> LayerNorm epilogue of the columns [cb, cb + H/2) of one row.  ONE pass over TMEM: a = act(z) goes to
// the image as fp16 hi / lo (22 bits); the two statistics passes and the normalisation then run over the thread's own image
// row in shared memory (cheap) instead of over TMEM, and xhat * XS overwrites a in place.
// `mid()` is called once the first half of this thread's columns holds the final xhat (both threads of a row reach it together:
// columns [0, H/4) and [H/2, 3H/4)), so that the MMA issuer can start the k-chunks of the next GEMM that read them while
// the other half is still being normalised.
struct NoMid { __device__ __forceinline__ void operator()() const {} };
template <int ACT, typename Mid = NoMid>
__device__ __forceinline__ void fwd_epilogue(int act_rt, uint32_t tacc, int H, const float* __restrict__ sbias, float descale,
                                             unsigned char* img, uint32_t img_bytes, int wch, const RowPair& P, float& mu, float& rstd,
                                             uint32_t (&mask)[2], Mid mid = Mid()) {
  const int r = P.r, nc = H >> 1, cb = P.half * nc;
  const float inv_n = 1.f / (float)H;
  uint32_t va[16], vb[16];
  float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
  uint32_t mk0 = 0u, mk1 = 0u;
  um::tmem_ld16_issue(tacc + cb, va);
#define HB_STEP(CC, CUR, NXT)                                                                              \
  if ((CC) * 16 < nc) {                                                                                    \
    um::tmem_ld_wait16(CUR);                                                                               \
    if (((CC) + 1) * 16 < nc) um::tmem_ld16_issue(tacc + cb + ((CC) + 1) * 16, NXT);                      \
    uint32_t m_ = 0u;                                                                                      \
    _Pragma("unroll") for (int q = 0; q < 2; ++q) {                                                        \
      const float4 ba = *reinterpret_cast<const float4*>(sbias + cb + (CC) * 16 + q * 8);                  \
      const float4 bb = *reinterpret_cast<const float4*>(sbias + cb + (CC) * 16 + q * 8 + 4);              \
      const float bq[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};                                \
      float x[8];                                                                                          \
      _Pragma("unroll") for (int j = 0; j < 8; ++j) {                                                      \
        const float z = fmaf(__uint_as_float(CUR[q * 8 + j]), descale, bq[j]);                             \
        m_ |= z > 0.f ? (1u << (q * 8 + j)) : 0u;                                                          \
        x[j] = act_f<ACT>(act_rt, z);                                                                      \
      }                                                                                                    \
      _Pragma("unroll") for (int j = 0; j < 8; j += 2) {                                                   \
        s0 += x[j]; s1 += x[j + 1];                                                                        \
        q0 = fmaf(x[j], x[j], q0); q1 = fmaf(x[j + 1], x[j + 1], q1);                                      \
      }                                                                                                    \
      uint4 hi, lo;                                                                                        \
      um::split8(x, hi, lo);                                                                               \
      const uint32_t off = img_off(r, (cb >> 3) + (CC) * 2 + q, wch);                                      \
      *reinterpret_cast<uint4*>(img + off) = hi;                                                           \
      *reinterpret_cast<uint4*>(img + img_bytes + off) = lo;                                               \
    }                                                                                                      \
    if ((CC) < 2) mk0 |= m_ << (16 * ((CC) & 1)); else mk1 |= m_ << (16 * ((CC) & 1));                     \
  }
  HB_STEP(0, va, vb) HB_STEP(1, vb, va) HB_STEP(2, va, vb) HB_STEP(3, vb, va)
#undef HB_STEP
  mask[0] = mk0; mask[1] = mk1;
  // statistics from one pass: var = E[a^2] - mean^2 (post-activation rows: var is the same order as E[a^2], the cancellation
  // costs a few ulp; a second pass over the row would double the fp16 -> fp32 conversions, the busiest pipe of this kernel)
  const float ps = s0 + s1, pq = q0 + q1;
  P.put(0, ps);
  P.put(1, pq);
  P.sync();
  mu = P.total(0, ps) * inv_n;
  rstd = rsqrtf(fmaxf(P.total(1, pq) * inv_n - mu * mu, 0.f) + 1e-5f);
  const float rs = rstd * XS, sh = -mu * rstd * XS;
  for (int c8 = 0; c8 < (nc >> 3); ++c8) {
    const uint32_t off = img_off(r, (cb >> 3) + c8, wch);
    float x[8];
    um::join8(*reinterpret_cast<const uint4*>(img + off), *reinterpret_cast<const uint4*>(img + img_bytes + off), x);
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = fmaf(x[j], rs, sh);
    uint4 hi, lo;
    um::split8(x, hi, lo);
    *reinterpret_cast<uint4*>(img + off) = hi;
    *reinterpret_cast<uint4*>(img + img_bytes + off) = lo;
    if (c8 == (nc >> 4) - 1) mid();
  }
}

// LayerNorm + activation backward of this thread's columns of one row: G = accumulator (= g / descale, g = dL/dxhat), x = XS * xhat
// from the image; writes DZS * dZ over xhat.  With s1 = sum G, s2 = sum G x:
//   dZ = rstd (g - mean(g) - xhat mean(g xhat)) act'   =   [rstd descale] (G - s1 / H - x s2 / (H XS^2)) act'
// `pre()` runs between the read-only statistics pass and the in-place write-back: the caller waits there for the MMAs that
// still READ this image (the weight-gradient GEMMs of the layer above, committed separately from the dX GEMM whose result
// this epilogue consumes), so those MMAs overlap the statistics pass instead of delaying the whole epilogue.
template <int ACT, typename Pre>
__device__ __forceinline__ void bwd_epilogue(int act_rt, uint32_t tacc, int H, float descale, unsigned char* img,
                                             uint32_t img_bytes, int wch, const RowPair& P, float mu, float rstd,
                                             const uint32_t (&mask)[2], bool row_ok, Pre pre) {
  const int r = P.r, nc = H >> 1, cb = P.half * nc;
  const float inv_n = 1.f / (float)H;
  // two passes over TMEM (sums, then the write-back): keeping the 64 accumulator values of a thread in registers across the
  // statistics exchange does not fit the 168-register cap of the 320-thread CTA next to the rest of the epilogue state
  float s1a = 0.f, s1b = 0.f, s2a = 0.f, s2b = 0.f;
  {
    uint32_t va[16], vb[16];
    um::tmem_ld16_issue(tacc + cb, va);
#define HB_STEP(CC, CUR, NXT)                                                                              \
    if ((CC) * 16 < nc) {                                                                                  \
      um::tmem_ld_wait16(CUR);                                                                             \
      if (((CC) + 1) * 16 < nc) um::tmem_ld16_issue(tacc + cb + ((CC) + 1) * 16, NXT);                    \
      _Pragma("unroll") for (int q = 0; q < 2; ++q) {                                                      \
        const uint32_t off = img_off(r, (cb >> 3) + (CC) * 2 + q, wch);                                    \
        float x[8];                                                                                        \
        um::join8(*reinterpret_cast<const uint4*>(img + off), *reinterpret_cast<const uint4*>(img + img_bytes + off), x); \
        _Pragma("unroll") for (int j = 0; j < 8; j += 2) {                                                 \
          const float g0 = __uint_as_float(CUR[q * 8 + j]), g1 = __uint_as_float(CUR[q * 8 + j + 1]);      \
          s1a += g0; s1b += g1;                                                                            \
          s2a = fmaf(g0, x[j], s2a); s2b = fmaf(g1, x[j + 1], s2b);                                        \
        }                                                                                                  \
      }                                                                                                    \
    }
    HB_STEP(0, va, vb) HB_STEP(1, vb, va) HB_STEP(2, va, vb) HB_STEP(3, vb, va)
#undef HB_STEP
  }
  const float p1 = s1a + s1b, p2 = s2a + s2b;
  P.put(0, p1);
  P.put(1, p2);
  P.sync();
  const float m1 = P.total(0, p1) * inv_n, m2 = P.total(1, p2) * inv_n * (1.f / (XS * XS));
  const float stdx = 1.f / (rstd * XS);
  const float k = row_ok ? rstd * descale * DZS : 0.f;
  pre();
  for (int cc = 0; cc * 16 < nc; ++cc) {
    uint32_t v[16];
    um::tmem_ld16_issue(tacc + cb + cc * 16, v);
    um::tmem_ld_wait16(v);
    const uint32_t mw = (cc < 2 ? mask[0] : mask[1]) >> (16 * (cc & 1));
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const uint32_t off = img_off(r, (cb >> 3) + cc * 2 + q, wch);
      float x[8], dz[8];
      um::join8(*reinterpret_cast<const uint4*>(img + off), *reinterpret_cast<const uint4*>(img + img_bytes + off), x);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float a = fmaf(x[j], stdx, mu);
        const float t = fmaf(-x[j], m2, __uint_as_float(v[q * 8 + j]) - m1);
        dz[j] = k * t * act_prime<ACT>(act_rt, a, (mw >> (q * 8 + j)) & 1u);
      }
      uint4 hi, lo;
      um::split8(dz, hi, lo);
      *reinterpret_cast<uint4*>(img + off) = hi;
      *reinterpret_cast<uint4*>(img + img_bytes + off) = lo;
    }
  }
}

__device__ __forceinline__ float huber_v(float e, float d, int use_huber, float* de) {
  if (!use_huber) { *de = e; return e * e / 2.f; }
  const float ae = fabsf(e);
  if (ae <= d) { *de = e; return e * e / 2.f; }
  *de = e > 0.f ? d : -d;
  return d * (ae - d / 2.f);
}

// Phase clock (profiling aid, HB_FUSED_TIMING=1): thread 64 of every CTA adds the SM-clock cycles it spends in each
// epilogue phase / each wait for the MMA warp to a global table, read back through hb_fused_timing_read.
__device__ unsigned long long g_phase_cycles[148 * 16];
__device__ int g_phase_on;
struct PhaseClock {   // accumulates in shared memory (a global read-modify-write per lap would itself cost ~600 cycles)
  unsigned long long t;
  unsigned long long* acc;
  bool on;
  __device__ __forceinline__ void start(bool enable, unsigned long long* smem_acc) {
    on = enable; acc = smem_acc;
    if (on) { for (int i = 0; i < 16; ++i) acc[i] = 0ull; t = clock64(); }
  }
  __device__ __forceinline__ void lap(int slot) {
    if (on) { const unsigned long long n = clock64(); acc[slot] += n - t; t = n; }
  }
  __device__ __forceinline__ void flush() {
    if (on) for (int i = 0; i < 16; ++i) g_phase_cycles[blockIdx.x * 16 + i] += acc[i];
  }
};

// ------------------------------------------------------------------------------------------------ the kernel
template <int HEAD, int MODE, int ACT>
__global__ void __launch_bounds__(THREADS, 1) fused_update_kernel(const __grid_constant__ Args a) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int H = a.H, K0p = a.K0p;
  const int wch0 = K0p >> 3, wchx = 16, wchd = NH >> 3, wchh = H >> 3;   // 8-feature chunks per image row
  const uint32_t x0_bytes = TILE * K0p * 2, x_bytes = TILE * 128 * 2, dl_bytes = TILE * NH * 2, wh_bytes = NH * H * 2;
  unsigned char* p = smem;
  unsigned char* X0 = p; p += 2 * x0_bytes;
  unsigned char* X1 = p; p += 2 * x_bytes;
  unsigned char* X2 = p; p += 2 * x_bytes;
  unsigned char* DL = p; p += 2 * dl_bytes;
  unsigned char* ONES = p; p += dl_bytes;
  unsigned char* WH = p; p += 2 * wh_bytes;
  const int STAGES = K0p <= 32 ? 3 : 2;
  unsigned char* ring = p; p += STAGES * STAGE_BYTES;
  float* sb0 = reinterpret_cast<float*>(p); p += 128 * 4;
  float* sb1 = reinterpret_cast<float*>(p); p += 128 * 4;
  float* sbh = reinterpret_cast<float*>(p); p += NH * 4;
  float* sstd = reinterpret_cast<float*>(p); p += 4 * NH * 4;       // Box: std, log std, d std / d log_std param, 1 / var
  float* sacc = reinterpret_cast<float*>(p); p += 2 * NH * 4;       // end-of-kernel sums: head bias grads, log_std grads
  double* sred = reinterpret_cast<double*>(p); p += 4 * 4 * 8;
  float* xch = reinterpret_cast<float*>(p); p += 2 * TILE * 2 * 4;  // row-pair exchange of partial sums
  uint64_t* bars = reinterpret_cast<uint64_t*>(p); p += 12 * 8;
  unsigned long long* sclk = reinterpret_cast<unsigned long long*>(p); p += 16 * 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(p);
  uint64_t* w_full = bars;                // [STAGES] weight chunk landed
  uint64_t* w_empty = bars + MAX_STAGES;  // [STAGES] MMAs reading the chunk retired
  uint64_t* e2m = bars + 2 * MAX_STAGES;  // epilogue warps -> MMA warp (8 arrivals: lane 0 of every epilogue warp)
  uint64_t* m2e = e2m + 1;            // MMA warp -> epilogue warps (tcgen05.commit)
  uint64_t* obs_free = e2m + 2;       // MMA warp -> producer: the staging image of the next tile's observations is dead
  uint64_t* obs_full = e2m + 3;       // producer's bulk copy -> epilogue warps
  uint64_t* e2m_h = e2m + 4;          // epilogue warps -> MMA warp: the first column half of a forward epilogue is final
  uint64_t* m2e_b = e2m + 5;          // MMA warp -> epilogue warps: the weight-gradient MMAs that read an image have retired
  unsigned char* OBS = MODE == M_GRAD ? X2 : X1;   // staging buffer = an activation image that is idle at that point
  const uint32_t obs_bytes = (uint32_t)TILE * (uint32_t)a.in_dim * 4u;
  // per-row inputs of the head phase ride along in the same staging image, behind the observation block (byte offsets; 0 = absent)
  const int aw = HEAD == HB_HEAD_BOX ? a.out : 1;
  uint32_t so = obs_bytes, o_act = 0, o_old = 0, o_adv = 0, o_fac = 0, o_w = 0, o_av = 0, o_vp = 0, o_ret = 0;
  if (HEAD != HB_HEAD_VALUE) {
    o_act = so; so += TILE * aw * 4;
    if (MODE == M_GRAD) {
      o_old = so; so += TILE * aw * 4;
      o_adv = so; so += TILE * 4;
      if (a.factor) { o_fac = so; so += TILE * 4; }
      if (a.use_active) { o_w = so; so += TILE * 4; }
    }
    if (HEAD == HB_HEAD_DISCRETE && a.avail != nullptr) { o_av = so; so += TILE * a.out * 4; }
  } else if (MODE == M_GRAD) {
    o_vp = so; so += TILE * 4;
    o_ret = so; so += TILE * 4;
  }
  const uint32_t stage_bytes = so;

  const long long ntiles = (a.rows + TILE - 1) / TILE;
  const int nch1 = H >> 5;
  constexpr bool GRAD = MODE == M_GRAD;

  // ---- one-time setup
  if (H < 128) {   // feature columns >= H of the activation images are read by the M = 128 weight-gradient MMAs, never written
    for (int i = tid; i < (int)((2 * x_bytes) / 16); i += THREADS) {
      reinterpret_cast<uint4*>(X1)[i] = make_uint4(0, 0, 0, 0);
      reinterpret_cast<uint4*>(X2)[i] = make_uint4(0, 0, 0, 0);
    }
  }
  for (int i = tid; i < TILE * 2; i += THREADS)   // ONES[row][16]: column 0 = 1.0, 16-byte chunks [row/8][2][row%8]
    reinterpret_cast<uint4*>(ONES)[i] = ((i >> 3) & 1) ? make_uint4(0, 0, 0, 0) : make_uint4(0x00003C00u, 0, 0, 0);
  for (int i = tid; i < (int)((2 * wh_bytes) / 16); i += THREADS) reinterpret_cast<uint4*>(WH)[i] = reinterpret_cast<const uint4*>(a.imgh)[i];
  for (int i = tid; i < 128; i += THREADS) { sb0[i] = i < H ? a.bias0[i] : 0.f; sb1[i] = i < H ? a.bias1[i] : 0.f; }
  if (tid < NH) {
    sbh[tid] = a.biash[tid];
    sacc[tid] = sacc[NH + tid] = 0.f;
    float sd = 1.f, ls = 0.f, dsd = 0.f;
    if (HEAD == HB_HEAD_BOX && tid < a.out) {
      const float sig = 1.f / (1.f + expf(-a.log_std[tid] / a.std_x));
      sd = sig * a.std_y;
      ls = logf(sd);
      dsd = a.std_y * sig * (1.f - sig) / a.std_x;
    }
    sstd[tid] = sd; sstd[NH + tid] = ls; sstd[2 * NH + tid] = dsd; sstd[3 * NH + tid] = 1.f / (sd * sd);
  }
  if (tid < 16) sred[tid] = 0.0;
  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) { um::mbar_init(&w_full[i], 1); um::mbar_init(&w_empty[i], 1); }
    um::mbar_init(e2m, 8);             // one arrival per epilogue warp
    um::mbar_init(e2m_h, 8);
    um::mbar_init(m2e_b, 1);
    um::mbar_init(m2e, 1);
    um::mbar_init(obs_free, 1);
    um::mbar_init(obs_full, 1);
    um::fence_mbarrier_init();
  }
  if (warp == 0) um::tmem_alloc(tmem_slot, TMEM_COLS);
  um::fence_async_smem();
  um::tc_fence_before();
  __syncthreads();
  um::tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const float ws0 = a.scales[0], ws1 = a.scales[1], wsh = a.scales[2];

  if (warp == 0) {
    // ================================================================ weight-chunk producer (one lane)
    if (lane == 0) {
      uint32_t it = 0, tl_ = 0;
      auto staged = [&](long long t) { return a.stage_obs && t < ntiles && (t + 1) * TILE <= a.rows; };
      auto load_obs = [&](long long t) {
        um::mbar_expect_tx(obs_full, stage_bytes);
        um::tma_bulk_g2s(OBS, a.obs + t * TILE * a.in_dim, obs_bytes, obs_full);
        const long long r0 = t * TILE;
        if (o_act) um::tma_bulk_g2s(OBS + o_act, a.actions + r0 * aw, TILE * aw * 4, obs_full);
        if (o_old) um::tma_bulk_g2s(OBS + o_old, a.old_logp + r0 * aw, TILE * aw * 4, obs_full);
        if (o_adv) um::tma_bulk_g2s(OBS + o_adv, a.adv + r0, TILE * 4, obs_full);
        if (o_fac) um::tma_bulk_g2s(OBS + o_fac, a.factor + r0, TILE * 4, obs_full);
        if (o_w) um::tma_bulk_g2s(OBS + o_w, a.active + r0, TILE * 4, obs_full);
        if (o_av) um::tma_bulk_g2s(OBS + o_av, a.avail + r0 * a.out, TILE * a.out * 4, obs_full);
        if (o_vp) um::tma_bulk_g2s(OBS + o_vp, a.value_preds + r0, TILE * 4, obs_full);
        if (o_ret) um::tma_bulk_g2s(OBS + o_ret, a.returns + r0, TILE * 4, obs_full);
      };
      if (staged(blockIdx.x)) load_obs(blockIdx.x);
      for (long long t = blockIdx.x; t < ntiles; t += gridDim.x, ++tl_) {
        for (int pass = 0; pass < (GRAD ? 3 : 2); ++pass) {
          const int layer = pass == 0 ? 0 : 1;
          const int nch = layer == 0 ? a.nch0 : nch1, kp = layer == 0 ? K0p : H;
          const unsigned char* src = reinterpret_cast<const unsigned char*>(pass == 0 ? a.img0 : (pass == 1 ? a.img1 : a.img1b));
          for (int ci = 0; ci < nch; ++ci, ++it) {
            // layer-1 forward at H = 128: the k-chunks of the two column quarters that are final first (0, 2) go first
            const int c = (pass == 1 && nch == 4) ? ((ci & 1) * 2 + (ci >> 1)) : ci;
            const int kc = kp - 32 * c < 32 ? kp - 32 * c : 32;
            const uint32_t bytes = 2u * (uint32_t)H * (uint32_t)kc * 2u;
            const uint32_t st = it % STAGES, use = it / STAGES;
            if (use > 0) um::mbar_wait(&w_empty[st], (use - 1) & 1);
            um::mbar_expect_tx(&w_full[st], bytes);
            um::tma_bulk_g2s(ring + st * STAGE_BYTES, src + (size_t)c * (2u * H * 32u * 2u), bytes, &w_full[st]);
          }
        }
        // the staging image is free once this tile's MMAs that read it have retired: fetch the next tile's observations
        um::mbar_wait(obs_free, tl_ & 1);
        if (staged(t + gridDim.x)) load_obs(t + gridDim.x);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================================================ MMA issuer (one lane)
    if (lane == 0) {
      uint32_t it = 0, pe = 0, peh = 0;
      bool first = true;
      const uint32_t X0a = um::smem_u32(X0), X1a = um::smem_u32(X1), X2a = um::smem_u32(X2), DLa = um::smem_u32(DL);
      const uint32_t ONa = um::smem_u32(ONES), WHa = um::smem_u32(WH), RGa = um::smem_u32(ring);
      for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
        auto wait_e = [&]() { um::mbar_wait(e2m, pe); pe ^= 1; um::tc_fence_after(); };
        auto wait_eh = [&]() { um::mbar_wait(e2m_h, peh); peh ^= 1; um::tc_fence_after(); };
        auto chunk = [&](int kc, auto&& body) {   // consume the next ring stage
          const uint32_t st = it % STAGES, use = it / STAGES;
          um::mbar_wait(&w_full[st], use & 1);
          um::tc_fence_after();
          body(RGa + st * STAGE_BYTES, (uint32_t)H * (uint32_t)kc * 2u);
          um::commit(&w_empty[st]);
          ++it;
        };
        // -- layer 0: C_F = X0 W0'^T
        wait_e();
        for (int c = 0; c < a.nch0; ++c) {
          const int kc = K0p - 32 * c < 32 ? K0p - 32 * c : 32;
          chunk(kc, [&](uint32_t wb, uint32_t wimg) {
            gemm3(tmem + C_F, op_kmajor(X0a, x0_bytes, wch0, 4 * c), op_kmajor(wb, wimg, kc >> 3, 0), kc >> 4,
                  um::idesc_f16(H, 0, 0), c > 0);
          });
        }
        um::commit(m2e);
        // -- layer 1: C_F = X1 W1'^T.  H = 128: the k-chunks of the column quarters [0, 32) and [64, 96) start as soon as the
        // layer-0 epilogue has finalised them (e2m_h), the other two when it is done (the ring delivers them in that order)
        wait_eh();
        if (nch1 == 4) {
          auto l1 = [&](int c, bool acc) {
            chunk(32, [&](uint32_t wb, uint32_t wimg) {
              gemm3(tmem + C_F, op_kmajor(X1a, x_bytes, wchx, 4 * c), op_kmajor(wb, wimg, 4, 0), 2, um::idesc_f16(H, 0, 0), acc);
            });
          };
          l1(0, false); l1(2, true);
          wait_e();
          l1(1, true); l1(3, true);
        } else {
          wait_e();
          for (int c = 0; c < nch1; ++c)
            chunk(32, [&](uint32_t wb, uint32_t wimg) {
              gemm3(tmem + C_F, op_kmajor(X1a, x_bytes, wchx, 4 * c), op_kmajor(wb, wimg, 4, 0), 2, um::idesc_f16(H, 0, 0), c > 0);
            });
        }
        um::commit(m2e);
        if (!GRAD) um::commit(obs_free);   // evaluate: X1 (the staging image) is dead after these MMAs
        // -- head: C_H = X2 Wh'^T (same split over the column quarters of the layer-1 epilogue)
        wait_eh();
        if (H == 128) {
          auto hd = [&](int q, bool acc) {
            gemm3(tmem + C_H, op_kmajor(X2a, x_bytes, wchx, 4 * q), op_kmajor(WHa, wh_bytes, wchh, 4 * q), 2, um::idesc_f16(NH, 0, 0), acc);
          };
          hd(0, false); hd(2, true);
          wait_e();
          hd(1, true); hd(3, true);
        } else {
          wait_e();
          gemm3(tmem + C_H, op_kmajor(X2a, x_bytes, wchx, 0), op_kmajor(WHa, wh_bytes, wchh, 0), H >> 4, um::idesc_f16(NH, 0, 0), false);
        }
        um::commit(m2e);
        if (GRAD) {
          // -- head backward: C_F = DL Wh' (dL/dxhat_1);  C_WH += X2^T DL
          wait_e();
          gemm3(tmem + C_F, op_kmajor(DLa, dl_bytes, wchd, 0), op_mnmajor(WHa, wh_bytes, wchh, 0), 1, um::idesc_f16(H, 0, 1), false);
          um::commit(m2e);                 // the layer-1 backward epilogue only needs C_F; the sums below still READ X2 and DL
          gemm3(tmem + C_WH, op_mnmajor(X2a, x_bytes, wchx, 0), op_mnmajor(DLa, dl_bytes, wchd, 0), TILE >> 4,
                um::idesc_f16(NH, 1, 1), !first);
          // column sums of DL over the rows: M = 128 reads past the 16 real columns (finite garbage in lanes >= 16, unused)
          gemm3(tmem + C_BH, op_mnmajor(DLa, dl_bytes, wchd, 0), op_mnmajor(ONa, dl_bytes, wchd, 0), TILE >> 4,
                um::idesc_f16(NH, 1, 1), !first, false);
          um::commit(m2e_b);               // ... the epilogue waits for this one before it overwrites X2
          // -- layer 1 backward: C_W1 += dZ1^T X1;  C_B1 += dZ1^T 1;  C_F = dZ1 W1' (dL/dxhat_0), one weight chunk at a time
          wait_e();
          // the chunks already sitting in the ring go first, so their stages are released (and refilled by the producer)
          // while the weight-gradient MMAs, which need no streamed operand, run
          // dX accumulates over chunks of 32 output features n: A = dZ1[:, 32c .. 32c+32) (K-major), B = W1'[32c .. 32c+32)[:]
          // as an MN-major operand (N = h input features) -- full-width MMAs, every operand byte read once
          auto dx_chunk = [&](int c) {
            chunk(32, [&](uint32_t wb, uint32_t wimg) {
              gemm3(tmem + C_F, op_kmajor(X2a, x_bytes, wchx, 4 * c), op_mnmajor(wb, wimg, H >> 3, 0), 2,
                    um::idesc_f16(H, 0, 1), c > 0);
            });
          };
          // the bias column sums (small) run while the last weight chunk streams in; the big weight-gradient GEMM goes AFTER the
          // commit that releases the layer-0 backward epilogue (which needs only C_F) and is waited for separately (m2e_b)
          const int nres = nch1 < STAGES ? nch1 : STAGES;
          for (int c = 0; c < nres; ++c) dx_chunk(c);
          gemm3(tmem + C_B1, op_mnmajor(X2a, x_bytes, wchx, 0), op_mnmajor(ONa, dl_bytes, wchd, 0), TILE >> 4,
                um::idesc_f16(NH, 1, 1), !first, false);
          for (int c = nres; c < nch1; ++c) dx_chunk(c);
          um::commit(m2e);
          gemm3(tmem + C_W1, op_mnmajor(X2a, x_bytes, wchx, 0), op_mnmajor(X1a, x_bytes, wchx, 0), TILE >> 4,
                um::idesc_f16(H, 1, 1), !first);
          um::commit(m2e_b);
          um::commit(obs_free);            // X2 (the staging image) is dead after these MMAs
          // -- layer 0 backward: C_W0 += dZ0^T X0;  C_B0 += dZ0^T 1
          wait_e();
          gemm3(tmem + C_W0, op_mnmajor(X1a, x_bytes, wchx, 0), op_mnmajor(X0a, x0_bytes, wch0, 0), TILE >> 4,
                um::idesc_f16(K0p, 1, 1), !first);
          gemm3(tmem + C_B0, op_mnmajor(X1a, x_bytes, wchx, 0), op_mnmajor(ONa, dl_bytes, wchd, 0), TILE >> 4,
                um::idesc_f16(NH, 1, 1), !first, false);
          um::commit(m2e);
          first = false;
        }
      }
    }
    __syncwarp();
  } else {
    // ================================================================ epilogue warps: thread = row
    // warps 2-5: column half 0, warps 6-9: column half 1 of the same rows (TMEM lane quarter = warp % 4)
    const int q = warp & 3, r = q * 32 + lane, half = (warp - 2) >> 2;
    const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16);
    const RowPair RP{xch, half, r, 2 + q};
    uint32_t pm = 0, po = 0;
    auto wait_m = [&]() { um::mbar_wait(m2e, pm); pm ^= 1; um::tc_fence_after(); };
    auto signal = [&]() { um::fence_async_smem(); um::tc_fence_before(); __syncwarp(); if (lane == 0) um::mbar_arrive(e2m); };
    auto mid = [&]() { um::fence_async_smem(); um::tc_fence_before(); __syncwarp(); if (lane == 0) um::mbar_arrive(e2m_h); };
    uint32_t pmb = 0;
    auto wait_mb = [&]() { um::mbar_wait(m2e_b, pmb); pmb ^= 1; um::tc_fence_after(); };
    const int na = a.out;
    float s_loss = 0.f, s_ent = 0.f, s_ratio = 0.f, s_rows = 0.f;
    float vmean = 0.f, vstd = 1.f;
    if (HEAD == HB_HEAD_VALUE && a.vn_state != nullptr) {  // valuenorm.py:38-45
      const float d = fmaxf(a.vn_state[2], 1e-5f);
      const float mu = a.vn_state[0] / d, msq = a.vn_state[1] / d;
      vmean = mu;
      vstd = sqrtf(fmaxf(msq - mu * mu, 1e-2f));
    }
    bool pending = false;   // a backward MMA group of the previous tile may still read X0 / X1
    PhaseClock pc;
    pc.start(g_phase_on != 0 && tid == 64, sclk);   // warp 2, lane 0: a half-0 thread
    for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
      const long long row = t * TILE + r;
      const bool ok = row < a.rows;
      const bool ld = ok && half == 0;   // the column-half-0 thread of a row owns its inputs, the head and the loss
      const long long src = ld ? (a.index ? (long long)a.index[row] : row) : 0;
      // full tiles: the producer's bulk copies put the 128 x in_dim observation block and the per-row inputs of the head phase
      // into the (idle) staging image; partial / gathered tiles read global memory directly
      const bool st_obs = a.stage_obs && (t + 1) * TILE <= a.rows;
      if (st_obs && half == 0) { um::mbar_wait(obs_full, po); po ^= 1; }
      const float* stg = reinterpret_cast<const float*>(OBS);
      const long long si = st_obs ? r : src;     // row index into the staged block / the global array
      auto in = [&](const float* g, uint32_t off) -> const float* { return st_obs ? stg + (off >> 2) : g; };
      // ---- per-row inputs of the head phase, read now (the staging image is rewritten by the layer epilogues)
      float in_act = 0.f, in_old = 0.f, in_adv = 0.f, in_fac = 1.f, in_w = 1.f, in_vp = 0.f, in_ret = 0.f;
      float in_actv[HEAD == HB_HEAD_BOX ? 8 : 1], in_oldv[HEAD == HB_HEAD_BOX ? 8 : 1];
      unsigned in_avm = 0xffffu;
      if (HEAD == HB_HEAD_DISCRETE) {
        if (ld) {
          in_act = in(a.actions, o_act)[si];
          if (GRAD) {
            in_old = in(a.old_logp, o_old)[si]; in_adv = in(a.adv, o_adv)[si];
            if (a.factor) in_fac = in(a.factor, o_fac)[si];
            if (a.use_active) in_w = in(a.active, o_w)[si];
          }
          if (a.avail != nullptr) {
            const float* av = in(a.avail, o_av) + si * a.out;
            in_avm = 0u;
#pragma unroll
            for (int j = 0; j < NH; ++j) in_avm |= (j < a.out && av[j < a.out ? j : 0] != 0.f) ? (1u << j) : 0u;
          }
        }
      } else if (HEAD == HB_HEAD_BOX) {
#pragma unroll
        for (int j = 0; j < (HEAD == HB_HEAD_BOX ? 8 : 1); ++j) {
          in_actv[j] = (ld && j < a.out) ? in(a.actions, o_act)[si * a.out + j] : 0.f;
          in_oldv[j] = (ld && GRAD && j < a.out) ? in(a.old_logp, o_old)[si * a.out + j] : 0.f;
        }
        if (ld && GRAD) {
          in_adv = in(a.adv, o_adv)[si];
          if (a.factor) in_fac = in(a.factor, o_fac)[si];
          if (a.use_active) in_w = in(a.active, o_w)[si];
        }
      } else if (ld && GRAD) {
        in_vp = in(a.value_preds, o_vp)[si]; in_ret = in(a.returns, o_ret)[si];
      }
      (void)in_vp; (void)in_ret; (void)in_act; (void)in_old; (void)in_actv; (void)in_oldv;
      // next tile's rows -> L2 (identity index only): the first touch of a tile then costs an L2 hit, not a DRAM round trip
      {
        const long long tn = t + gridDim.x;
        const long long rown = tn * TILE + r;
        if (!a.stage_obs && a.index == nullptr && rown < a.rows && half == 0) {
          if (!a.stage_obs) {
            const float* on = a.obs + rown * a.in_dim;
            um::prefetch_l2(on);
            um::prefetch_l2(on + a.in_dim - 1);
          }
          if (lane == 0) {
            if (HEAD == HB_HEAD_VALUE) { if (GRAD) { um::prefetch_l2(a.value_preds + rown); um::prefetch_l2(a.returns + rown); } }
            else {
              if (HEAD == HB_HEAD_DISCRETE) um::prefetch_l2(a.actions + rown);
              if (GRAD) {
                um::prefetch_l2(a.adv + rown);
                if (HEAD == HB_HEAD_DISCRETE) um::prefetch_l2(a.old_logp + rown);
                if (a.factor) um::prefetch_l2(a.factor + rown);
                if (a.use_active) um::prefetch_l2(a.active + rown);
              }
            }
          }
          if (HEAD == HB_HEAD_DISCRETE && a.avail != nullptr) um::prefetch_l2(a.avail + rown * a.out);
          if (HEAD == HB_HEAD_BOX) { um::prefetch_l2(a.actions + rown * a.out); if (GRAD) um::prefetch_l2(a.old_logp + rown * a.out); }
        }
      }
      // ---- feature LayerNorm of the observation row (mlp.py:57-66), exact two-pass statistics; the row sits in registers
      const float* o = st_obs ? stg + r * a.in_dim : a.obs + src * a.in_dim;
      float mean = 0.f, rs = 0.f;
      if (half == 0) {
        float s = 0.f;
        for (int k0 = 0; k0 < a.in_dim; k0 += 16) {
          float x[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) x[j] = (ld && k0 + j < a.in_dim) ? o[k0 + j] : 0.f;
#pragma unroll
          for (int j = 0; j < 16; ++j) s += x[j];
        }
        mean = s / (float)a.in_dim;
        float qv = 0.f;
        for (int k0 = 0; k0 < a.in_dim; k0 += 16) {
          float x[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) x[j] = (ld && k0 + j < a.in_dim) ? o[k0 + j] : 0.f;
#pragma unroll
          for (int j = 0; j < 16; ++j) { const float d = x[j] - mean; qv = k0 + j < a.in_dim ? fmaf(d, d, qv) : qv; }
        }
        rs = rsqrtf(qv / (float)a.in_dim + 1e-5f);
      }
      pc.lap(0);                                   // inputs + feature-norm statistics
      if (pending) { wait_m(); pending = false; }
      pc.lap(1);                                   // wait: last backward MMAs of the previous tile
      const float rsx = rs * XS;
      if (half == 0) {
        for (int k0 = 0; k0 < K0p; k0 += 16) {
          float x[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) x[j] = (ld && k0 + j < a.in_dim) ? (o[k0 + j] - mean) * rsx : 0.f;
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const float xc[8] = {x[c * 8], x[c * 8 + 1], x[c * 8 + 2], x[c * 8 + 3], x[c * 8 + 4], x[c * 8 + 5], x[c * 8 + 6], x[c * 8 + 7]};
            uint4 hi, lo;
            um::split8(xc, hi, lo);
            const uint32_t off = img_off(r, (k0 >> 3) + c, wch0);
            *reinterpret_cast<uint4*>(X0 + off) = hi;
            *reinterpret_cast<uint4*>(X0 + x0_bytes + off) = lo;
          }
        }
      }
      signal();
      pc.lap(2);                                   // X0 image written
      // ---- layer 0
      float mu0, rstd0, mu1, rstd1;
      uint32_t mask0[2] = {0, 0}, mask1[2] = {0, 0};
      wait_m();
      pc.lap(3);                                   // wait: layer-0 MMAs
      fwd_epilogue<ACT>(a.act, tl + C_F, H, sb0, 1.f / (XS * ws0), X1, x_bytes, wchx, RP, mu0, rstd0, mask0, mid);
      signal();
      pc.lap(4);                                   // layer-0 epilogue
      // ---- layer 1
      wait_m();
      pc.lap(5);                                   // wait: layer-1 MMAs
      fwd_epilogue<ACT>(a.act, tl + C_F, H, sb1, 1.f / (XS * ws1), X2, x_bytes, wchx, RP, mu1, rstd1, mask1, mid);
      signal();
      pc.lap(6);                                   // layer-1 epilogue
      // ---- head
      wait_m();
      pc.lap(7);                                   // wait: head MMAs
      float dl[NH];
#pragma unroll
      for (int j = 0; j < NH; ++j) dl[j] = 0.f;
      if (half == 0) {
        float hv[NH];
        um::tmem_ld16(tl + C_H, hv);
        const float hdesc = 1.f / (XS * wsh);
        if (HEAD == HB_HEAD_DISCRETE) {
          float lg[NH], lp[NH], pj[NH];
#pragma unroll
          for (int j = 0; j < NH; ++j) lg[j] = hv[j] * hdesc;
          const unsigned avm = in_avm;
          const float ent = rows::categorical<NH>(lg, sbh, na, avm, lp, pj);
          const int act = ld ? (int)in_act : 0;
          const float lpa = rows::select<NH>(lp, act);
          if (MODE == M_EVAL) {
            if (ok) {
              if (a.logp_out) a.logp_out[row] = lpa;
              if (a.factor_inout) a.factor_inout[src] = a.factor_inout[src] * expf(lpa - a.logp_ref[src]);
            }
          } else {
            // happo.py:66-91 (the 1 / sum(active) normaliser is applied when the slots are reduced)
            const float w = in_w, fac = in_fac, adv = in_adv, old = in_old;
            const float ratio = expf(lpa - old);
            float m;
            const float dm = dmin_dratio(ratio, adv, a.clip, a.use_clip, &m);
            const float okf = ok ? 1.f : 0.f;
            if (ok && a.logp_out) a.logp_out[row] = lpa;     // the log-probs under the weights of this pass, for free
            const float c_lp = -fac * w * dm * ratio * okf;
            const float c_h = a.entropy_coef * w * okf;
            if (ok) { s_loss += -fac * m * w; s_ent += ent * w; s_ratio += ratio; s_rows += 1.f; }
#pragma unroll
            for (int j = 0; j < NH; ++j) {
              const bool live = j < na && ((avm >> j) & 1u);
              dl[j] = live ? c_lp * ((j == act ? 1.f : 0.f) - pj[j]) + c_h * pj[j] * (lp[j] + ent) : 0.f;
            }
          }
        } else if (HEAD == HB_HEAD_BOX) {
          // DiagGaussian (distributions.py:24-34,58-89)
          float lpj[NH], dlt[NH];
          float ent_row = 0.f;
#pragma unroll
          for (int j = 0; j < NH; ++j) {
            lpj[j] = 0.f; dlt[j] = 0.f;
            if (j < na) {
              const float mean_j = fmaf(hv[j], hdesc, sbh[j]);
              dlt[j] = (j < 8 ? in_actv[HEAD == HB_HEAD_BOX ? (j < 8 ? j : 0) : 0] : 0.f) - mean_j;
              lpj[j] = -(dlt[j] * dlt[j]) * 0.5f * sstd[3 * NH + j] - sstd[NH + j] - 0.5f * HB_LOG_2PI_F;
              ent_row += 0.5f + 0.5f * HB_LOG_2PI_F + sstd[NH + j];
            }
          }
          if (MODE == M_EVAL) {
            if (ok) {
              float agg = a.agg_prod ? 1.f : 0.f;
#pragma unroll
              for (int j = 0; j < NH; ++j) {
                if (j < na) {
                  if (a.logp_out) a.logp_out[row * na + j] = lpj[j];
                  if (a.factor_inout) {
                    const float e = expf(lpj[j] - a.logp_ref[src * na + j]);
                    agg = a.agg_prod ? agg * e : agg + e;
                  }
                }
              }
              if (a.factor_inout) a.factor_inout[src] = a.factor_inout[src] * (a.agg_prod ? agg : agg / (float)na);
            }
          } else {
            const float w = in_w, fac = in_fac, adv = in_adv;
            if (ok && a.logp_out) {
#pragma unroll
              for (int j = 0; j < NH; ++j)
                if (j < na) a.logp_out[row * na + j] = lpj[j];
            }
            float e[NH];
            float ratio = a.agg_prod ? 1.f : 0.f;
#pragma unroll
            for (int j = 0; j < NH; ++j) {
              e[j] = 0.f;
              if (j < na) {
                e[j] = expf(lpj[j] - (j < 8 ? in_oldv[HEAD == HB_HEAD_BOX ? (j < 8 ? j : 0) : 0] : 0.f));
                ratio = a.agg_prod ? ratio * e[j] : ratio + e[j];
              }
            }
            if (!a.agg_prod) ratio /= (float)na;
            float m;
            const float dm = dmin_dratio(ratio, adv, a.clip, a.use_clip, &m);
            const float okf = ok ? 1.f : 0.f;
            const float c_r = -fac * w * dm * okf;
            if (ok) { s_loss += -fac * m * w; s_ent += ent_row * w; s_ratio += ratio; s_rows += 1.f; }
#pragma unroll
            for (int j = 0; j < NH; ++j) {
              if (j < na) {
                const float sd = sstd[j], ivar = sstd[3 * NH + j];
                const float c_lp = c_r * (a.agg_prod ? ratio : e[j] / (float)na);
                const float dmean = c_lp * dlt[j] * ivar;
                const float dstd = c_lp * (dlt[j] * dlt[j] * ivar / sd - 1.f / sd) - a.entropy_coef * w * okf / sd;
                dl[j] = dmean;
                if (j < 8) dl[8 + j] = dstd * sstd[2 * NH + j];   // d loss / d log_std[j]: summed over rows by the C_BH MMAs
              }
            }
          }
        } else {
          // value head + cal_value_loss (v_critic.py:75-114); the 1 / rows normaliser is applied at the slot reduction
          const float v = fmaf(hv[0], hdesc, sbh[0]);
          if (MODE == M_EVAL) {
            if (ok && a.logp_out) a.logp_out[row] = v;
          } else {
            const float vp = in_vp;
            float ret = in_ret;
            if (a.vn_state != nullptr) ret = (ret - vmean) / vstd;
            const float dv = v - vp;
            const float dc = fminf(fmaxf(dv, -a.clip), a.clip);
            const float vclip = vp + dc;
            const bool pass = dv >= -a.clip && dv <= a.clip;
            float de_c, de_o;
            const float l_c = huber_v(ret - vclip, a.huber_delta, a.use_huber, &de_c);
            const float l_o = huber_v(ret - v, a.huber_delta, a.use_huber, &de_o);
            const float g_o = -de_o, g_c = pass ? -de_c : 0.f;
            float loss = l_o, g = g_o;
            if (a.use_clipped) {
              if (l_c > l_o) { loss = l_c; g = g_c; }
              else if (l_c == l_o) { loss = l_o; g = 0.5f * (g_o + g_c); }
            }
            g = ok ? g * a.vcoef : 0.f;
            if (ok) { s_loss += loss; s_rows += 1.f; }
            dl[0] = g;
          }
        }
      }
      if (!GRAD) continue;   // evaluate: nothing of this tile is read by a later MMA group
      if (half == 0) {
        float x[8];
        uint4 hi, lo;
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
#pragma unroll
          for (int j = 0; j < 8; ++j) x[j] = dl[ch * 8 + j] * DZS;
          um::split8(x, hi, lo);
          const uint32_t off = img_off(r, ch, wchd);
          *reinterpret_cast<uint4*>(DL + off) = hi;
          *reinterpret_cast<uint4*>(DL + dl_bytes + off) = lo;
        }
      }
      signal();
      pc.lap(8);                                   // head epilogue (loss, d logits)
      // ---- layer 1 backward (dL/dxhat_1 in C_F), dZ_1 over xhat_1 in X2
      wait_m();
      pc.lap(9);                                   // wait: head backward MMAs
      bwd_epilogue<ACT>(a.act, tl + C_F, H, 1.f / (DZS * wsh), X2, x_bytes, wchx, RP, mu1, rstd1, mask1, ok, wait_mb);
      signal();
      pc.lap(10);                                  // layer-1 backward epilogue
      // ---- layer 0 backward (dL/dxhat_0 in C_F), dZ_0 over xhat_0 in X1
      wait_m();
      pc.lap(11);                                  // wait: layer-1 backward MMAs (dW1, db1, dX through 4 weight chunks)
      bwd_epilogue<ACT>(a.act, tl + C_F, H, 1.f / (DZS * ws1), X1, x_bytes, wchx, RP, mu0, rstd0, mask0, ok, wait_mb);
      signal();
      pc.lap(12);                                  // layer-0 backward epilogue
      pending = true;
    }
    if (GRAD && pending) wait_m();
    pc.flush();
    if (GRAD && half == 0) {
      // ---- flush: this CTA's weight-gradient sums -> its slot of the split buffer (lane = output feature n)
      float* slot = a.part + (long long)blockIdx.x * a.part_stride;
      const int n = r;
      for (int c0 = 0; c0 < H; c0 += 32) {
        float v[32];
        um::tmem_ld32(tl + C_W1 + c0, v);
        if (n < H) {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(slot + a.pw1 + n * H + c0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      }
      for (int c0 = 0; c0 < K0p; c0 += 16) {
        float v[16];
        um::tmem_ld16(tl + C_W0 + c0, v);
        if (n < H) {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (c0 + j < a.in_dim) slot[a.pw0 + n * a.in_dim + c0 + j] = v[j];
        }
      }
      {
        float v[16];
        um::tmem_ld16(tl + C_B1, v);
        if (n < H) slot[a.pb1 + n] = v[0];
        um::tmem_ld16(tl + C_B0, v);
        if (n < H) slot[a.pb0 + n] = v[0];
        um::tmem_ld16(tl + C_WH, v);
        if (n < H) {
#pragma unroll
          for (int j = 0; j < NH; ++j)
            if (j < na) slot[a.phw + j * H + n] = v[j];
        }
      }
      {
        float v[16];
        um::tmem_ld16(tl + C_BH, v);
        if (n < na) slot[a.phb + n] = v[0];
        if (HEAD == HB_HEAD_BOX && n >= 8 && n < 8 + na) slot[a.plogstd + n - 8] = v[0];
      }
      // the loss scalars: sums over this CTA's rows
      const double d0 = warp_sum_d((double)s_loss), d1 = warp_sum_d((double)s_ent), d2 = warp_sum_d((double)s_ratio), d3 = warp_sum_d((double)s_rows);
      if (lane == 0) { sred[q * 4 + 0] = d0; sred[q * 4 + 1] = d1; sred[q * 4 + 2] = d2; sred[q * 4 + 3] = d3; }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (r < 4) {
        const double s = sred[r] + sred[4 + r] + sred[8 + r] + sred[12 + r];
        if (HEAD == HB_HEAD_VALUE) { if (r == 0) atomicAdd(a.scalars, s); if (r == 3) atomicAdd(a.scalars + 1, s); }
        else atomicAdd(a.scalars + r, s);
      }
    }
  }
  um::tc_fence_before();
  __syncthreads();
  if (warp == 0) um::tmem_dealloc(tmem, TMEM_COLS);
}


// ================================================================================================ rollout inference
// One launch per rollout step for every actor and the critic (OnPolicyBaseRunner.collect, on_policy_base_runner.py:285-340):
// CTA = one 128-row tile of one net; the same tcgen05 forward as the update kernel (feature norm -> 2 x [MMA, act + LayerNorm
// epilogue] -> head MMA) followed by the sampling head (Philox4x32-10 keyed exactly like the FP32 kernels it replaces:
// fused_infer.cu / rowwise.cu) or the value head.  Replaces the FP32 FFMA fused_infer_kernel for the shapes the fused kernel covers.
constexpr uint32_t ACT_TMEM_COLS = 256;

template <int ACT>
__global__ void __launch_bounds__(THREADS, 1) fused_act_kernel(const __grid_constant__ ActArgs A) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  int ni = 0;
  for (int q = 1; q < A.n_nets; ++q) if ((int)blockIdx.x >= A.net[q].tile0) ni = q;
  const ActNet& N = A.net[ni];
  const long long t = (long long)blockIdx.x - N.tile0;
  const int H = A.H, K0p = N.K0p;
  const int wch0 = K0p >> 3, wchx = 16, wchh = H >> 3;
  const uint32_t x0_bytes = TILE * A.K0p_max * 2, x_bytes = TILE * 128 * 2, wh_bytes = NH * H * 2;
  unsigned char* p = smem;
  unsigned char* X0 = p; p += 2 * x0_bytes;
  unsigned char* X1 = p; p += 2 * x_bytes;
  unsigned char* X2 = p; p += 2 * x_bytes;
  unsigned char* WH = p; p += 2 * wh_bytes;
  unsigned char* ring = p; p += 2 * STAGE_BYTES;
  float* sb0 = reinterpret_cast<float*>(p); p += 128 * 4;
  float* sb1 = reinterpret_cast<float*>(p); p += 128 * 4;
  float* sbh = reinterpret_cast<float*>(p); p += NH * 4;
  float* xch = reinterpret_cast<float*>(p); p += 2 * TILE * 2 * 4;
  uint64_t* bars = reinterpret_cast<uint64_t*>(p); p += 8 * 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(p);
  uint64_t* w_full = bars;        // [2]
  uint64_t* w_empty = bars + 2;   // [2]
  uint64_t* e2m = bars + 4;
  uint64_t* m2e = bars + 5;
  uint64_t* obs_full = bars + 6;
  unsigned char* OBS = X2;        // staging image: idle until the layer-1 epilogue
  constexpr int STG = 2;
  const __half* img0 = reinterpret_cast<const __half*>(N.prep + N.o_w0);
  const __half* img1 = reinterpret_cast<const __half*>(N.prep + N.o_w1);
  const int nch1 = H >> 5;
  const bool full = (t + 1) * TILE <= N.rows;
  const bool st_obs = N.stage && full;
  const uint32_t obs_bytes = (uint32_t)TILE * (uint32_t)N.in_dim * 4u;
  const uint32_t o_av = (N.head == HB_HEAD_DISCRETE && N.avail != nullptr) ? obs_bytes : 0u;
  const uint32_t stage_bytes = obs_bytes + (o_av ? (uint32_t)TILE * N.out * 4u : 0u);

  if (H < 128) {
    for (int i = tid; i < (int)((2 * x_bytes) / 16); i += THREADS) {
      reinterpret_cast<uint4*>(X1)[i] = make_uint4(0, 0, 0, 0);
      reinterpret_cast<uint4*>(X2)[i] = make_uint4(0, 0, 0, 0);
    }
  }
  for (int i = tid; i < (int)((2 * wh_bytes) / 16); i += THREADS)
    reinterpret_cast<uint4*>(WH)[i] = reinterpret_cast<const uint4*>(N.prep + N.o_hw)[i];
  for (int i = tid; i < 128; i += THREADS) { sb0[i] = i < H ? N.prep[N.o_b0 + i] : 0.f; sb1[i] = i < H ? N.prep[N.o_b1 + i] : 0.f; }
  if (tid < NH) sbh[tid] = N.prep[N.o_bh + tid];
  if (tid == 0) {
    for (int i = 0; i < STG; ++i) { um::mbar_init(&w_full[i], 1); um::mbar_init(&w_empty[i], 1); }
    um::mbar_init(e2m, 8);
    um::mbar_init(m2e, 1);
    um::mbar_init(obs_full, 1);
    um::fence_mbarrier_init();
  }
  if (warp == 0) um::tmem_alloc(tmem_slot, ACT_TMEM_COLS);
  um::fence_async_smem();
  um::tc_fence_before();
  __syncthreads();
  um::tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const float ws0 = N.prep[N.o_sc], ws1 = N.prep[N.o_sc + 1], wsh = N.prep[N.o_sc + 2];

  if (warp == 0) {
    if (lane == 0) {
      if (st_obs) {
        um::mbar_expect_tx(obs_full, stage_bytes);
        um::tma_bulk_g2s(OBS, N.obs + t * TILE * N.in_dim, obs_bytes, obs_full);
        if (o_av) um::tma_bulk_g2s(OBS + o_av, N.avail + t * TILE * N.out, TILE * N.out * 4, obs_full);
      }
      uint32_t it = 0;
      for (int pass = 0; pass < 2; ++pass) {
        const int nch = pass == 0 ? N.nch0 : nch1, kp = pass == 0 ? K0p : H;
        const unsigned char* src = reinterpret_cast<const unsigned char*>(pass == 0 ? img0 : img1);
        for (int c = 0; c < nch; ++c, ++it) {
          const int kc = kp - 32 * c < 32 ? kp - 32 * c : 32;
          const uint32_t bytes = 2u * (uint32_t)H * (uint32_t)kc * 2u;
          const uint32_t st = it % STG, use = it / STG;
          if (use > 0) um::mbar_wait(&w_empty[st], (use - 1) & 1);
          um::mbar_expect_tx(&w_full[st], bytes);
          um::tma_bulk_g2s(ring + st * STAGE_BYTES, src + (size_t)c * (2u * H * 32u * 2u), bytes, &w_full[st]);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      uint32_t it = 0, pe = 0;
      const uint32_t X0a = um::smem_u32(X0), X1a = um::smem_u32(X1), X2a = um::smem_u32(X2), WHa = um::smem_u32(WH), RGa = um::smem_u32(ring);
      auto wait_e = [&]() { um::mbar_wait(e2m, pe); pe ^= 1; um::tc_fence_after(); };
      auto chunk = [&](int kc, auto&& body) {
        const uint32_t st = it % STG, use = it / STG;
        um::mbar_wait(&w_full[st], use & 1);
        um::tc_fence_after();
        body(RGa + st * STAGE_BYTES, (uint32_t)H * (uint32_t)kc * 2u);
        um::commit(&w_empty[st]);
        ++it;
      };
      wait_e();
      for (int c = 0; c < N.nch0; ++c) {
        const int kc = K0p - 32 * c < 32 ? K0p - 32 * c : 32;
        chunk(kc, [&](uint32_t wb, uint32_t wimg) {
          gemm3(tmem + C_F, op_kmajor(X0a, x0_bytes, wch0, 4 * c), op_kmajor(wb, wimg, kc >> 3, 0), kc >> 4, um::idesc_f16(H, 0, 0), c > 0);
        });
      }
      um::commit(m2e);
      wait_e();
      for (int c = 0; c < nch1; ++c)
        chunk(32, [&](uint32_t wb, uint32_t wimg) {
          gemm3(tmem + C_F, op_kmajor(X1a, x_bytes, wchx, 4 * c), op_kmajor(wb, wimg, 4, 0), 2, um::idesc_f16(H, 0, 0), c > 0);
        });
      um::commit(m2e);
      wait_e();
      gemm3(tmem + 128, op_kmajor(X2a, x_bytes, wchx, 0), op_kmajor(WHa, wh_bytes, wchh, 0), H >> 4, um::idesc_f16(NH, 0, 0), false);
      um::commit(m2e);
    }
    __syncwarp();
  } else {
    const int q = warp & 3, r = q * 32 + lane, half = (warp - 2) >> 2;
    const uint32_t tl = tmem + ((uint32_t)(q * 32) << 16);
    const RowPair RP{xch, half, r, 2 + q};
    uint32_t pm = 0;
    auto wait_m = [&]() { um::mbar_wait(m2e, pm); pm ^= 1; um::tc_fence_after(); };
    auto signal = [&]() { um::fence_async_smem(); um::tc_fence_before(); __syncwarp(); if (lane == 0) um::mbar_arrive(e2m); };
    const long long row = t * TILE + r;
    const bool ok = row < N.rows;
    const bool ld = ok && half == 0;
    const int na = N.out;
    if (st_obs && half == 0) um::mbar_wait(obs_full, 0);
    const float* stg = reinterpret_cast<const float*>(OBS);
    unsigned avm = 0xffffu;
    if (N.head == HB_HEAD_DISCRETE && N.avail != nullptr && ld) {
      const float* av = st_obs ? stg + (o_av >> 2) + r * na : N.avail + row * na;
      avm = 0u;
#pragma unroll
      for (int j = 0; j < NH; ++j) avm |= (j < na && av[j < na ? j : 0] != 0.f) ? (1u << j) : 0u;
    }
    const float* o = st_obs ? stg + r * N.in_dim : N.obs + (ok ? row : 0) * N.in_dim;
    float mean = 0.f, rs = 0.f;
    if (half == 0) {
      float s = 0.f;
      for (int k0 = 0; k0 < N.in_dim; k0 += 16) {
        float x[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) x[j] = (ld && k0 + j < N.in_dim) ? o[k0 + j] : 0.f;
#pragma unroll
        for (int j = 0; j < 16; ++j) s += x[j];
      }
      mean = s / (float)N.in_dim;
      float qv = 0.f;
      for (int k0 = 0; k0 < N.in_dim; k0 += 16) {
        float x[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) x[j] = (ld && k0 + j < N.in_dim) ? o[k0 + j] : 0.f;
#pragma unroll
        for (int j = 0; j < 16; ++j) { const float d = x[j] - mean; qv = k0 + j < N.in_dim ? fmaf(d, d, qv) : qv; }
      }
      rs = rsqrtf(qv / (float)N.in_dim + 1e-5f);
      const float rsx = rs * XS;
      for (int k0 = 0; k0 < K0p; k0 += 16) {
        float x[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) x[j] = (ld && k0 + j < N.in_dim) ? (o[k0 + j] - mean) * rsx : 0.f;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const float xc[8] = {x[c * 8], x[c * 8 + 1], x[c * 8 + 2], x[c * 8 + 3], x[c * 8 + 4], x[c * 8 + 5], x[c * 8 + 6], x[c * 8 + 7]};
          uint4 hi, lo;
          um::split8(xc, hi, lo);
          const uint32_t off = img_off(r, (k0 >> 3) + c, wch0);
          *reinterpret_cast<uint4*>(X0 + off) = hi;
          *reinterpret_cast<uint4*>(X0 + x0_bytes + off) = lo;
        }
      }
    }
    signal();
    float mu0, rstd0, mu1, rstd1;
    uint32_t mask0[2], mask1[2];
    wait_m();
    fwd_epilogue<ACT>(A.act, tl + C_F, H, sb0, 1.f / (XS * ws0), X1, x_bytes, wchx, RP, mu0, rstd0, mask0);
    signal();
    wait_m();
    fwd_epilogue<ACT>(A.act, tl + C_F, H, sb1, 1.f / (XS * ws1), X2, x_bytes, wchx, RP, mu1, rstd1, mask1);
    signal();
    wait_m();
    if (half == 0) {
      float hv[NH];
      um::tmem_ld16(tl + 128, hv);
      const float hdesc = 1.f / (XS * wsh);
      const unsigned long long off = A.offset + (A.offset_base ? *A.offset_base : 0ull);
      if (N.head == HB_HEAD_VALUE) {
        if (ok) N.out0[row] = fmaf(hv[0], hdesc, sbh[0]);
      } else if (N.head == HB_HEAD_DISCRETE) {
        float lg[NH], lp[NH], pj[NH];
#pragma unroll
        for (int j = 0; j < NH; ++j) lg[j] = hv[j] * hdesc;
        rows::categorical<NH>(lg, sbh, na, avm, lp, pj);
        const int pick = rows::categorical_pick<NH>(pj, na, A.deterministic != 0, A.deterministic ? 0.f : rows::row_uniform(row, N.seed, off));
        const float lpp = rows::select<NH>(lp, pick);
        if (ok) { N.out0[row] = (float)pick; N.out1[row] = lpp; }
      } else {
        const float* log_std = N.prep + N.o_ls;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (j < na) {
            const float mean_j = fmaf(hv[j], hdesc, sbh[j]);
            const float sig = 1.f / (1.f + expf(-log_std[j] / N.std_x));
            const float sd = sig * N.std_y, lsd = logf(sd);
            float act = mean_j;
            if (!A.deterministic) {
              const uint4 rnd = philox4x32(make_uint4((uint32_t)row, (uint32_t)((unsigned long long)row >> 32), (uint32_t)j, (uint32_t)off),
                                           make_uint2((uint32_t)N.seed, (uint32_t)(N.seed >> 32) ^ (uint32_t)(off >> 32)));
              const float u1 = u01(rnd.x), u2 = u01(rnd.y);
              act = mean_j + sd * (sqrtf(-2.f * logf(u1)) * cospif(2.f * u2));
            }
            if (ok) {
              const float dv = act - mean_j;
              N.out0[row * na + j] = act;
              N.out1[row * na + j] = -(dv * dv) / (2.f * sd * sd) - lsd - 0.5f * HB_LOG_2PI_F;
            }
          }
        }
      }
    }
  }
  um::tc_fence_before();
  __syncthreads();
  if (warp == 0) um::tmem_dealloc(tmem, ACT_TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------ weight images
// One launch per weight matrix: W'[n][k] = W[n][k] * gamma[k], scaled by a power of two so that max |W'| lands in
// [128, 256), split into fp16 hi / lo, written as KC-wide k-chunks of K-major core matrices; folded bias b' = b + W beta.
struct PackJob {
  const float* W; const float* gamma; const float* beta; const float* b;
  int N, K, Nimg, Kp, KC, RC;
  __half* img; float* bias_out; float* scale_out;
  int cta0, ctas;          // this job's CTA range in the launch
};
struct PackJobs { PackJob j[4]; int n; };

__global__ void __launch_bounds__(256) fused_pack_kernel(PackJobs jobs) {
  __shared__ float smax[8];
  __shared__ float sscale;
  int ji = 0;
  for (int q = 1; q < jobs.n; ++q) if ((int)blockIdx.x >= jobs.j[q].cta0) ji = q;
  const PackJob& J = jobs.j[ji];
  const int cta = blockIdx.x - J.cta0;
  const float* __restrict__ W = J.W;
  const float* __restrict__ gamma = J.gamma;
  const int N = J.N, K = J.K, Nimg = J.Nimg, Kp = J.Kp, KC = J.KC, RC = J.RC;
  __half* __restrict__ img = J.img;
  float mx = 0.f;
  for (int i = threadIdx.x; i < N * K; i += 256) mx = fmaxf(mx, fabsf(W[i] * (gamma ? gamma[i % K] : 1.f)));
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) smax[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = 0.f;
    for (int i = 0; i < 8; ++i) m = fmaxf(m, smax[i]);
    int ex = 0;
    if (m > 0.f) frexpf(m, &ex);                     // m = f * 2^ex, f in [0.5, 1)
    ex = ex < -20 ? -20 : (ex > 20 ? 20 : ex);
    sscale = m > 0.f ? exp2f((float)(8 - ex)) : 1.f;
    if (cta == 0 && J.scale_out != nullptr) *J.scale_out = sscale;
  }
  __syncthreads();
  const float sc = sscale;
  const int total = Nimg * Kp;
  for (int i = cta * 256 + threadIdx.x; i < total; i += J.ctas * 256) {
    const int n = i / Kp, k = i % Kp;
    const float v = (n < N && k < K) ? W[n * K + k] * (gamma ? gamma[k] : 1.f) * sc : 0.f;
    const __half hi = __float2half_rn(v);
    const __half lo = __float2half_rn(v - __half2float(hi));
    if (RC > 0) {   // chunks of RC rows, each a [RC][Kp] K-major image pair (hi, lo)
      const int c = n / RC, nl = n % RC;
      const size_t chunk0 = (size_t)c * (2u * RC * Kp);
      const size_t e = (size_t)((nl >> 3) * (Kp >> 3) + (k >> 3)) * 64 + (nl & 7) * 8 + (k & 7);
      img[chunk0 + e] = hi;
      img[chunk0 + (size_t)RC * Kp + e] = lo;
      continue;
    }
    const int c = k / KC, kl = k % KC;                                          // KC-wide k-chunks (the last may be narrower)
    const int kc = Kp - KC * c < KC ? Kp - KC * c : KC;
    const size_t chunk0 = (size_t)c * (2u * Nimg * KC);                        // halves before this chunk
    const size_t e = (size_t)((n >> 3) * (kc >> 3) + (kl >> 3)) * 64 + (n & 7) * 8 + (kl & 7);
    img[chunk0 + e] = hi;
    img[chunk0 + (size_t)Nimg * kc + e] = lo;
  }
  if (J.bias_out != nullptr) {   // b' = b + W beta: one warp per output row (coalesced reads of the row), rows over the job's CTAs
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int n = cta * 8 + warp; n < Nimg; n += J.ctas * 8) {
      float v = 0.f;
      if (n < N && J.beta)
        for (int k = lane; k < K; k += 32) v += W[n * K + k] * J.beta[k];
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) J.bias_out[n] = n < N ? J.b[n] + v : 0.f;
    }
  }
}

// ------------------------------------------------------------------------------------------------ slot reduction
struct Regions { int n; int off[8]; int len[8]; float scale[8]; };
// grad[i] = scale_i * norm * sum over the CTA slots.  A CTA owns 32 consecutive parameters; warp g sums slot group g (every load
// of a warp is one coalesced 128-byte line, 16 loads of a thread in flight at once), the groups are added in order by
// warp 0: deterministic, two memory round trips instead of slots / 16.  <= 42 registers x 256 threads so that the CTA fits
// on an SM next to a CTA of the other stream's persistent update kernel.
constexpr int SR_GROUPS = 8, SR_MAXPER = 16;
__global__ void __launch_bounds__(32 * SR_GROUPS, 6) fused_slot_reduce_kernel(float* __restrict__ grad, const float* __restrict__ part, int slots,
                                                                           long long stride, int total, const __grid_constant__ Regions R,
                                                                           const double* __restrict__ norm3, double host_scale) {
  __shared__ float sm[SR_GROUPS][32];
  const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  const int per = (slots + SR_GROUPS - 1) / SR_GROUPS;
  const int s0 = g * per, s1 = s0 + per < slots ? s0 + per : slots;
  float acc = 0.f;
  if (i < total) {
    for (int sb = s0; sb < s1; sb += SR_MAXPER) {
      float v[SR_MAXPER];
#pragma unroll
      for (int u = 0; u < SR_MAXPER; ++u) v[u] = sb + u < s1 ? part[(long long)(sb + u) * stride + i] : 0.f;
#pragma unroll
      for (int u = 0; u < SR_MAXPER; ++u) acc += v[u];
    }
  }
  sm[g][lane] = acc;
  __syncthreads();
  if (g != 0 || i >= total) return;
  float sc = 0.f;
  bool in = false;
  for (int q = 0; q < R.n; ++q)
    if (i >= R.off[q] && i < R.off[q] + R.len[q]) { sc = R.scale[q]; in = true; }
  if (!in) { grad[i] = 0.f; return; }
  float t = 0.f;
#pragma unroll
  for (int q = 0; q < SR_GROUPS; ++q) t += sm[q][lane];
  const double nrm = host_scale * (norm3 ? 1.0 / norm3[2] : 1.0);
  grad[i] = (float)((double)t * (double)sc * nrm);
}

// LayerNorm-affine unfolding for every consumer (layer 0 / layer 1 / head) in one launch: one warp per input column k.
//   G = d/dW', gb = d/db' (in the W / b slots of grad):  dgamma[k] = sum_n W[n][k] G[n][k],  dbeta[k] = sum_n W[n][k] gb[n],
//   dW[n][k] = gamma[k] G[n][k] + beta[k] gb[n],  db = gb      (optim.cu featnorm_grad_fold_kernel, warp-parallel over n)
struct Folds { int n; int w[3], b[3], gw[3], gb[3], N[3], K[3], col0[3]; };
__global__ void __launch_bounds__(128) fused_unfold_kernel(const float* __restrict__ params, float* __restrict__ grad, Folds F, int cols) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= cols) return;
  int f = 0;
  for (int q = 1; q < F.n; ++q) if (warp >= F.col0[q]) f = q;
  const int k = warp - F.col0[f], N = F.N[f], K = F.K[f];
  const float gam = params[F.gw[f] + k], bet = params[F.gb[f] + k];
  double dg = 0.0, dbt = 0.0;
  for (int n = lane; n < N; n += 32) {
    const float w = params[F.w[f] + n * K + k];
    const float G = grad[F.w[f] + n * K + k];
    const float gb = grad[F.b[f] + n];
    dg += (double)w * (double)G;
    dbt += (double)w * (double)gb;
    grad[F.w[f] + n * K + k] = fmaf(gam, G, bet * gb);
  }
  dg = warp_sum_d(dg);
  dbt = warp_sum_d(dbt);
  if (lane == 0) { grad[F.gw[f] + k] = (float)dg; grad[F.gb[f] + k] = (float)dbt; }
}

static std::atomic<int> g_enabled{-1};

}  // namespace fz

// profiling aid: enable / read the per-phase cycle table of the fused kernel (out: [148][16] uint64)
int fused_timing_enable(int on) {
  static const unsigned long long zeros[148 * 16] = {0};
  cudaError_t e = cudaMemcpyToSymbol(fz::g_phase_cycles, zeros, sizeof(zeros));
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(fz::g_phase_on, &on, sizeof(int));
  return e == cudaSuccess ? HB_OK : cuda_fail(e, "fused_timing_enable");
}
int fused_timing_read(unsigned long long* out) {
  cudaError_t e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpyFromSymbol(out, fz::g_phase_cycles, sizeof(unsigned long long) * 148 * 16);
  return e == cudaSuccess ? HB_OK : cuda_fail(e, "fused_timing_read");
}

bool fused_enabled() {
  int v = fz::g_enabled.load(std::memory_order_relaxed);
  if (v < 0) {
    const char* e = getenv("HB_FUSED");
    v = (e != nullptr && atoi(e) == 0) ? 0 : 1;
    fz::g_enabled.store(v);
  }
  return v != 0 && gemm_impl() != 0;   // HB_GEMM_IMPL=fp32 keeps every GEMM on the FP32 SIMT parity anchor
}
void set_fused_enabled(int v) { fz::g_enabled.store(v ? 1 : 0); }

bool fused_shape_ok(const hb_net_desc* d) {
  if (d->rnn_layers != 0 || d->n_layers != 2 || d->hidden[0] != d->hidden[1]) return false;
  const int H = d->hidden[0];
  if (H != 32 && H != 64 && H != 128) return false;
  if (!d->feature_norm || d->in_dim < 1 || d->in_dim > 64) return false;
  if (d->activation == HB_ACT_HARDSWISH) return false;
  if (d->out_dim < 1 || d->out_dim > (d->head == HB_HEAD_BOX ? 8 : fz::NH)) return false;
  return true;
}

int launch_fused_pack(const hb_net_desc* d, const ParamLayout& P, const PrepLayout& Q, const float* params, float* prepared,
                      cudaStream_t st) {
  const int H = d->hidden[0];
  float* sc = prepared + Q.fz_scale;
  fz::PackJobs jobs;
  memset(&jobs, 0, sizeof(jobs));
  int cta = 0;
  auto add = [&](const float* W, const float* g, const float* be, const float* b, int N, int K, int Nimg, int Kp, int KC, int RC,
                 float* img, float* bias_out, float* scale_out, int ctas) {
    fz::PackJob& J = jobs.j[jobs.n++];
    J.W = W; J.gamma = g; J.beta = be; J.b = b; J.N = N; J.K = K; J.Nimg = Nimg; J.Kp = Kp; J.KC = KC; J.RC = RC;
    J.img = reinterpret_cast<__half*>(img); J.bias_out = bias_out; J.scale_out = scale_out; J.cta0 = cta; J.ctas = ctas;
    cta += ctas;
  };
  add(params + P.w[0], params + P.fn_w, params + P.fn_b, params + P.b[0], H, d->in_dim, H, Q.fz_k0p, 32, 0, prepared + Q.fz_w[0],
      prepared + Q.fz_bias[0], sc + 0, 8);
  add(params + P.w[1], params + P.lnw[0], params + P.lnb[0], params + P.b[1], H, H, H, H, 32, 0, prepared + Q.fz_w[1],
      prepared + Q.fz_bias[1], sc + 1, 16);
  add(params + P.w[1], params + P.lnw[0], params + P.lnb[0], params + P.b[1], H, H, H, H, 32, 32, prepared + Q.fz_w1b, nullptr, nullptr, 16);
  add(params + P.hw, params + P.lnw[1], params + P.lnb[1], params + P.hbias, d->out_dim, H, fz::NH, H, H, 0, prepared + Q.fz_hw,
      prepared + Q.fz_hbias, sc + 2, 4);
  fz::fused_pack_kernel<<<cta, 256, 0, st>>>(jobs);
  HB_LAUNCH_DONE(st, "fused_pack");
  return HB_OK;
}


int fused_act_fill(fz::ActNet* n, const hb_net_desc* d, const float* prepared, const float* obs, const float* avail, float* out0,
                   float* out1, unsigned long long seed, long long rows, bool* ok) {
  PrepLayout Q;
  int rc = make_layouts(d, nullptr, &Q, nullptr);
  if (rc) return rc;
  *ok = Q.fz_ok != 0 && (d->head != HB_HEAD_BOX || d->out_dim <= 8);
  if (!*ok) return HB_OK;
  n->prep = prepared; n->obs = obs; n->avail = avail; n->out0 = out0; n->out1 = out1; n->seed = seed; n->rows = rows;
  n->in_dim = d->in_dim; n->out = d->out_dim; n->head = d->head; n->K0p = Q.fz_k0p; n->nch0 = Q.fz_chunks[0];
  n->o_w0 = Q.fz_w[0]; n->o_w1 = Q.fz_w[1]; n->o_hw = Q.fz_hw; n->o_b0 = Q.fz_bias[0]; n->o_b1 = Q.fz_bias[1]; n->o_bh = Q.fz_hbias;
  n->o_sc = Q.fz_scale; n->o_ls = Q.log_std; n->std_x = d->std_x_coef; n->std_y = d->std_y_coef;
  const uintptr_t bits = reinterpret_cast<uintptr_t>(obs) | reinterpret_cast<uintptr_t>(avail);
  n->stage = (bits & 15) == 0 ? 1 : 0;
  return HB_OK;
}

// A.n_nets, A.H, A.act, A.deterministic, A.offset(_base) and every net (fused_act_fill) set by the caller
int launch_fused_act(fz::ActArgs& A, cudaStream_t st) {
  int tiles = 0, k0 = 16;
  for (int i = 0; i < A.n_nets; ++i) {
    A.net[i].tile0 = tiles;
    tiles += (int)((A.net[i].rows + fz::TILE - 1) / fz::TILE);
    k0 = A.net[i].K0p > k0 ? A.net[i].K0p : k0;
  }
  A.K0p_max = k0;
  if (tiles == 0) return HB_OK;
  const size_t smem = 2 * (size_t)fz::TILE * k0 * 2 + 2 * 2 * (size_t)fz::TILE * 128 * 2 + 2 * (size_t)fz::NH * A.H * 2 + 2 * fz::STAGE_BYTES +
                      2 * 128 * 4 + fz::NH * 4 + 2 * fz::TILE * 2 * 4 + 8 * 8 + 16 + 1024;
#define HB_FZA(ACTV)                                                                                  \
  {                                                                                                   \
    auto kern = fz::fused_act_kernel<ACTV>;                                                           \
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);               \
    kern<<<tiles, fz::THREADS, smem, st>>>(A);                                                        \
  }
  if (A.act == HB_ACT_RELU) HB_FZA(HB_ACT_RELU)
  else if (A.act == HB_ACT_TANH) HB_FZA(HB_ACT_TANH)
  else HB_FZA(-1)
#undef HB_FZA
  HB_LAUNCH_DONE(st, "fused_act");
  return HB_OK;
}

size_t fused_smem_bytes(int H, int K0p) {
  size_t b = 2 * (size_t)fz::TILE * K0p * 2 + 2 * 2 * (size_t)fz::TILE * 128 * 2 + 3 * (size_t)fz::TILE * fz::NH * 2 +
             2 * (size_t)fz::NH * H * 2 + (size_t)(K0p <= 32 ? 3 : 2) * fz::STAGE_BYTES;
  b += 2 * 128 * 4 + fz::NH * 4 + 4 * fz::NH * 4 + 2 * fz::NH * 4 + 16 * 8 + 2 * fz::TILE * 2 * 4 + 10 * 8 + 16 * 8 + 16;
  return b + 1024;
}

template <int HEAD, int MODE>
static int launch_fused_act(const fz::Args& a, int grid, size_t smem, cudaStream_t st) {
#define HB_FZ(ACTV)                                                                                   \
  {                                                                                                   \
    auto kern = fz::fused_update_kernel<HEAD, MODE, ACTV>;                                            \
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);               \
    kern<<<grid, fz::THREADS, smem, st>>>(a);                                                         \
  }
  if (a.act == HB_ACT_RELU) HB_FZ(HB_ACT_RELU)
  else if (a.act == HB_ACT_TANH) HB_FZ(HB_ACT_TANH)
  else HB_FZ(-1)
#undef HB_FZ
  return HB_OK;
}

// mode 0 = gradient, 1 = evaluate.  Caller guarantees fused_shape_ok(d) and a packed `prepared` buffer.
int launch_fused_update(const hb_net_desc* d, const PrepLayout& Q, const ParamLayout& P, const float* prepared, fz::Args a, int mode,
                        int* grid_out, cudaStream_t st) {
  const int H = d->hidden[0];
  a.H = H; a.K0p = Q.fz_k0p; a.in_dim = d->in_dim; a.out = d->out_dim; a.act = d->activation; a.nch0 = Q.fz_chunks[0];
  a.img0 = reinterpret_cast<const __half*>(prepared + Q.fz_w[0]);
  a.img1 = reinterpret_cast<const __half*>(prepared + Q.fz_w[1]);
  a.img1b = reinterpret_cast<const __half*>(prepared + Q.fz_w1b);
  a.imgh = reinterpret_cast<const __half*>(prepared + Q.fz_hw);
  a.bias0 = prepared + Q.fz_bias[0]; a.bias1 = prepared + Q.fz_bias[1]; a.biash = prepared + Q.fz_hbias;
  a.scales = prepared + Q.fz_scale;
  a.log_std = prepared + Q.log_std; a.std_x = d->std_x_coef; a.std_y = d->std_y_coef;
  a.pw0 = P.w[0]; a.pb0 = P.b[0]; a.pw1 = P.w[1]; a.pb1 = P.b[1]; a.phw = P.hw; a.phb = P.hbias; a.plogstd = P.log_std;
  {
    const void* ptrs[] = {a.obs, a.actions, a.old_logp, a.adv, a.factor, a.active, a.avail, a.value_preds, a.returns};
    uintptr_t bits = 0;
    for (const void* q : ptrs) bits |= reinterpret_cast<uintptr_t>(q);
    a.stage_obs = (a.index == nullptr && (bits & 15) == 0) ? 1 : 0;   // TMA bulk copies need 16-byte aligned sources
  }
  const long long ntiles = (a.rows + fz::TILE - 1) / fz::TILE;
  const int grid = (int)(ntiles < 148 ? ntiles : 148);
  if (grid_out) *grid_out = grid;
  const size_t smem = fused_smem_bytes(H, Q.fz_k0p);
  int rc;
  if (d->head == HB_HEAD_DISCRETE) rc = mode == 0 ? launch_fused_act<HB_HEAD_DISCRETE, fz::M_GRAD>(a, grid, smem, st) : launch_fused_act<HB_HEAD_DISCRETE, fz::M_EVAL>(a, grid, smem, st);
  else if (d->head == HB_HEAD_BOX) rc = mode == 0 ? launch_fused_act<HB_HEAD_BOX, fz::M_GRAD>(a, grid, smem, st) : launch_fused_act<HB_HEAD_BOX, fz::M_EVAL>(a, grid, smem, st);
  else rc = mode == 0 ? launch_fused_act<HB_HEAD_VALUE, fz::M_GRAD>(a, grid, smem, st) : launch_fused_act<HB_HEAD_VALUE, fz::M_EVAL>(a, grid, smem, st);
  if (rc) return rc;
  HB_LAUNCH_DONE(st, shape_label(mode == 0 ? (d->head == HB_HEAD_VALUE ? "fused_critic_update" : "fused_actor_update") : "fused_evaluate",
                                 a.rows, H, d->in_dim));
  return HB_OK;
}

// slot sums -> grad (scaled), then the LayerNorm-affine unfolding per consumer (layer 0 / layer 1 / head)
int launch_fused_finish(const hb_net_desc* d, const ParamLayout& P, const float* params, float* grad, const float* part, int slots,
                        long long stride, const double* norm3, double host_scale, cudaStream_t st) {
  const int H = d->hidden[0];
  fz::Regions R;
  memset(&R, 0, sizeof(R));
  const float sw = 1.f / (fz::DZS * fz::XS), sb = 1.f / fz::DZS;
  int n = 0;
  auto add = [&](int off, int len, float s) { R.off[n] = off; R.len[n] = len; R.scale[n] = s; ++n; };
  add(P.w[0], H * d->in_dim, sw); add(P.b[0], H, sb);
  add(P.w[1], H * H, sw);         add(P.b[1], H, sb);
  add(P.hw, d->out_dim * H, sw);  add(P.hbias, d->out_dim, sb);
  if (d->head == HB_HEAD_BOX) add(P.log_std, d->out_dim, sb);
  R.n = n;
  fz::fused_slot_reduce_kernel<<<(P.total + 31) / 32, 32 * fz::SR_GROUPS, 0, st>>>(grad, part, slots, stride, P.total, R, norm3, host_scale);
  HB_LAUNCH_DONE(st, "fused_slot_reduce");
  fz::Folds F;
  memset(&F, 0, sizeof(F));
  int cols = 0;
  auto fold = [&](int w, int b, int gw, int gb, int N, int K) {
    const int q = F.n++;
    F.w[q] = w; F.b[q] = b; F.gw[q] = gw; F.gb[q] = gb; F.N[q] = N; F.K[q] = K; F.col0[q] = cols;
    cols += K;
  };
  fold(P.w[0], P.b[0], P.fn_w, P.fn_b, H, d->in_dim);
  fold(P.w[1], P.b[1], P.lnw[0], P.lnb[0], H, H);
  fold(P.hw, P.hbias, P.lnw[1], P.lnb[1], d->out_dim, H);
  fz::fused_unfold_kernel<<<(cols * 32 + 127) / 128, 128, 0, st>>>(params, grad, F, cols);
  HB_LAUNCH_DONE(st, "ln_affine_grad_fold");
  return HB_OK;
}

}  // namespace hb
