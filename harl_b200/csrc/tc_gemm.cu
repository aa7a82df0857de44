// tcgen05 (5th-gen tensor core) GEMM kernels with the LayerNorm epilogues of the MLP blocks (sm_100a).
//
//   tc_linear_ln_fwd : Y = LN(act(X W'^T + b'))     (same contract as the SIMT linear_ln_fwd_kernel)
//
// Numerics: kind::tf32 MMAs with fp32 accumulation in TMEM, error-compensated: x = hi + lo (hi = x rounded to TF32,
// lo = the residual rounded to TF32, both exactly representable in TF32 up to 2^-22) and
// D += A_hi B_hi + A_lo B_hi + A_hi B_lo, which restores fp32-level accuracy (relative error ~3e-7 per product) at
// 3 MMAs per k-step.
//
// Structure of one CTA (128 threads = 4 warps, one 128-row tile, UMMA 128 x NT x 8):
//   * operands live in shared memory in the canonical K-major no-swizzle UMMA layout
//       [row/8][k-chunk(4 floats)][row%8][4]   (LBO = 128 B between the two k-chunks of an MMA, SBO = 1024 B
//       between 8-row groups; a k-step of 8 advances the descriptor start by 256 B)
//   * B (weights) tiles are pre-packed in exactly that image by hb_net_prepare (hi image then lo image per
//     32-wide k-chunk), so one 1-D TMA bulk copy (cp.async.bulk ... mbarrier::complete_tx) stages a chunk;
//   * A (activation rows) are loaded by the 128 threads (one row each), split into hi/lo and stored;
//   * 2-stage ring: thread 0 issues the MMAs of a chunk and tcgen05.commit's the stage's `empty` mbarrier;
//   * accumulator rows are read back with tcgen05.ld.32x32b (thread t <-> TMEM lane t <-> tile row t), so the
//     LayerNorm row statistics are thread-local: three passes over TMEM (sum, centred sum of squares, write).
#include "common.cuh"
#include "kernels.cuh"
#include "umma.cuh"

namespace hb {

constexpr int TC_BM = 128;   // rows per CTA tile (UMMA_M)
constexpr int TC_KC = 32;    // floats of K per pipeline stage (4 MMA k-steps)
// One operand stage per CTA (64 KB at NT = 128 with the hi/lo images): three CTAs share an SM, so one CTA's global
// loads / epilogue overlap the others' MMAs -- inter-CTA instead of intra-CTA pipelining.
constexpr int TC_STAGES = 1;

// Round-to-nearest TF32 (cvt.rna): |x - hi| <= 2^-11 |x| and, for the residual, |r - lo| <= 2^-11 |r|, so
// x = hi + lo up to 2^-22 |x| -- four times tighter than clearing the low 13 mantissa bits, at the same MMA count.
// (two integer ops: add half a TF32 ulp to the magnitude bits, clear the low 13; a mantissa carry into the exponent
// is the correct round-up; inf / nan inputs are not preserved -- they are garbage in the reference as well.)
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u); }
__device__ __forceinline__ float tf32_lo(float x, float hi) { return tf32_hi(x - hi); }

// ------------------------------------------------------------------ weight tile packing (part of hb_net_prepare)
// Per job: for each k-chunk c (32 wide), hi image [NT][32] then lo image, canonical K-major UMMA layout;
// src(n, k) = W[n*ldn + k*ldk] * (scale ? scale[k] : 1), zero outside [N) x [K).
// All images of one net in ONE launch (blockIdx.y = job): hb_net_prepare runs after every optimiser step, and three
// 3-6 us launches per net were 2 % of the C2 update phase.
struct PackUmmaJobs {
  const float* W[2 * HB_MAX_LAYERS];
  const float* scale[2 * HB_MAX_LAYERS];
  float* dst[2 * HB_MAX_LAYERS];
  int ldn[2 * HB_MAX_LAYERS], ldk[2 * HB_MAX_LAYERS], N[2 * HB_MAX_LAYERS], K[2 * HB_MAX_LAYERS], NT[2 * HB_MAX_LAYERS],
      nchunks[2 * HB_MAX_LAYERS];
};
__global__ void pack_umma_jobs_kernel(const __grid_constant__ PackUmmaJobs J) {
  const int j = blockIdx.y;
  const float* __restrict__ W = J.W[j];
  const float* __restrict__ scale = J.scale[j];
  float* __restrict__ dst = J.dst[j];
  const int NT = J.NT[j], N = J.N[j], K = J.K[j], ldn = J.ldn[j], ldk = J.ldk[j];
  const int per_chunk = 2 * NT * TC_KC;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < J.nchunks[j] * NT * TC_KC; i += gridDim.x * blockDim.x) {
    const int c = i / (NT * TC_KC), e = i % (NT * TC_KC);
    // e indexes the image: [(n/8)][kc (8)][n%8][4]
    const int k4 = e & 3, n8 = (e >> 2) & 7, kc = (e >> 5) & 7, ng = e >> 8;
    const int n = ng * 8 + n8, k = c * TC_KC + kc * 4 + k4;
    float v = 0.f;
    if (n < N && k < K) { v = W[(int64_t)n * ldn + (int64_t)k * ldk]; if (scale) v *= scale[k]; }
    const float hi = tf32_hi(v);
    dst[(int64_t)c * per_chunk + e] = hi;
    dst[(int64_t)c * per_chunk + NT * TC_KC + e] = tf32_lo(v, hi);
  }
}

// jobs: (W, ldn, ldk, scale, N, K, NT, nchunks, dst) x njobs
int launch_pack_umma_jobs(int njobs, const float* const* W, const int* ldn, const int* ldk, const float* const* scale, const int* N,
                          const int* K, const int* NT, const int* nchunks, float* const* dst, cudaStream_t st) {
  if (njobs <= 0) return HB_OK;
  PackUmmaJobs J;
  int most = 0;
  for (int j = 0; j < njobs; ++j) {
    J.W[j] = W[j]; J.scale[j] = scale[j]; J.dst[j] = dst[j]; J.ldn[j] = ldn[j]; J.ldk[j] = ldk[j]; J.N[j] = N[j]; J.K[j] = K[j];
    J.NT[j] = NT[j]; J.nchunks[j] = nchunks[j];
    const int total = nchunks[j] * NT[j] * TC_KC;
    most = total > most ? total : most;
  }
  pack_umma_jobs_kernel<<<dim3((most + 255) / 256, njobs), 256, 0, st>>>(J);
  HB_LAUNCH_DONE(st, "pack_umma_tiles");
  return HB_OK;
}

int launch_pack_umma_tiles(const float* W, int ldn, int ldk, const float* scale, int N, int K, int NT, int nchunks,
                           float* dst, cudaStream_t st) {
  return launch_pack_umma_jobs(1, &W, &ldn, &ldk, &scale, &N, &K, &NT, &nchunks, &dst, st);
}

// ------------------------------------------------------------------ forward block on tcgen05
template <int NT>
struct TcSmem {
  float a[TC_STAGES][2][TC_BM * TC_KC];    // [stage][hi/lo] 16 KB each
  float b[TC_STAGES][2 * NT * TC_KC];      // [stage] hi image then lo image
  uint64_t full_b[TC_STAGES];              // TMA bytes landed
  uint64_t empty[TC_STAGES];               // MMAs that read the stage retired
  uint64_t done;                   // all MMAs retired
  uint32_t tmem_base;
  alignas(16) float pbias[NT];           // epilogue parameters (16-byte aligned: read as broadcast float4)
  alignas(16) float plnw[NT];
  alignas(16) float plnb[NT];
};

// One operand chunk of the mainloop: A = this thread's tile row from its first column of the chunk on (`k` of its 32
// columns are valid, the rest are staged as zeros), B = the chunk's pre-packed hi + lo weight image.
struct TcChunk {
  const float* a;
  int k;
  const float* b;
};

// Setup and mainloop shared by the forward, dX and tangent kernels: allocates NT TMEM columns and accumulates
// acc[128 x NT] = sum over n chunks of A_c B_c^T (3xTF32), with chunk(c) naming the operands of chunk c.  Returns the
// TMEM base address once every MMA has retired; the caller frees it with um::tmem_dealloc.
template <int NT, class ChunkOf>
__device__ __forceinline__ uint32_t tc_mainloop(TcSmem<NT>& s, int tid, bool row_ok, int n, ChunkOf&& chunk) {
  constexpr uint32_t B_BYTES = 2u * NT * TC_KC * sizeof(float);
  if (tid == 0) {
    for (int i = 0; i < TC_STAGES; ++i) { um::mbar_init(&s.full_b[i], 1); um::mbar_init(&s.empty[i], 1); }
    um::mbar_init(&s.done, 1);
    um::fence_mbarrier_init();
  }
  if ((tid >> 5) == 0) um::tmem_alloc(&s.tmem_base, NT);
  um::tc_fence_before();
  __syncthreads();
  um::tc_fence_after();
  const uint32_t tmem = s.tmem_base;
  constexpr uint32_t idesc = um::idesc_tf32(NT);

  uint32_t ph_full[2] = {0, 0}, ph_empty[2] = {0, 0};
  for (int c = 0; c < n; ++c) {
    const int st = c % TC_STAGES;
    if (c >= TC_STAGES) { um::mbar_wait(&s.empty[st], ph_empty[st]); ph_empty[st] ^= 1; }  // stage free again
    // chunk(c) is evaluated where each part is used: a B pointer formed outside the thread-0 branch costs every
    // thread two registers
    if (tid == 0) {
      um::mbar_expect_tx(&s.full_b[st], B_BYTES);
      um::tma_bulk_g2s(s.b[st], chunk(c).b, B_BYTES, &s.full_b[st]);
    }
    // A: thread t stages row t of the tile (zeros beyond M / the valid columns), hi and lo images
    {
      const TcChunk ch = chunk(c);
      float* ahi = s.a[st][0];
      float* alo = s.a[st][1];
      const int base = ((tid >> 3) * 8) * 32 + (tid & 7) * 4;  // floats: [(row/8)][kc][row%8][4]
#pragma unroll
      for (int kc = 0; kc < 8; ++kc) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row_ok && kc * 4 < ch.k) v = *reinterpret_cast<const float4*>(ch.a + kc * 4);
        float4 h = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
        *reinterpret_cast<float4*>(ahi + base + kc * 32) = h;
        *reinterpret_cast<float4*>(alo + base + kc * 32) = make_float4(tf32_lo(v.x, h.x), tf32_lo(v.y, h.y), tf32_lo(v.z, h.z), tf32_lo(v.w, h.w));
      }
    }
    um::fence_async_smem();   // generic-proxy smem writes -> visible to the tensor core (async proxy)
    __syncthreads();
    if (tid == 0) {
      um::mbar_wait(&s.full_b[st], ph_full[st]);
      um::tc_fence_after();
      const uint32_t a_hi = um::smem_u32(s.a[st][0]), a_lo = um::smem_u32(s.a[st][1]);
      const uint32_t b_hi = um::smem_u32(s.b[st]), b_lo = b_hi + NT * TC_KC * sizeof(float);
#pragma unroll
      for (int j = 0; j < TC_KC / 8; ++j) {
        const uint32_t off = j * 256;
        const uint64_t dah = um::desc(a_hi + off, 128, 1024), dbh = um::desc(b_hi + off, 128, 1024);
        um::mma_tf32(tmem, dah, dbh, idesc, (c | j) != 0);
        const uint64_t dal = um::desc(a_lo + off, 128, 1024), dbl = um::desc(b_lo + off, 128, 1024);
        um::mma_tf32(tmem, dal, dbh, idesc, 1);
        um::mma_tf32(tmem, dah, dbl, idesc, 1);
      }
      um::commit(&s.empty[st]);            // arrives when the MMAs above have finished reading this stage
      if (c == n - 1) um::commit(&s.done);
    }
    ph_full[st] ^= 1;
  }
  um::mbar_wait(&s.done, 0);
  um::tc_fence_after();
  return tmem;
}

template <int NT, int ACT>
__global__ void __launch_bounds__(128, 1) tc_linear_ln_fwd_kernel(const float* __restrict__ X, int ldx,
                                                                  const float* __restrict__ tiles, int nchunks,
                                                                  const float* __restrict__ bias,
                                                                  const float* __restrict__ lnw,
                                                                  const float* __restrict__ lnb, float* __restrict__ Z,
                                                                  float* __restrict__ Y, float* __restrict__ stats,
                                                                  int64_t M, int N, int Kred) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  TcSmem<NT>& s = *reinterpret_cast<TcSmem<NT>*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int64_t row0 = (int64_t)blockIdx.x * TC_BM;
  const int64_t row = row0 + tid;

  for (int i = tid; i < NT; i += 128) {
    s.pbias[i] = i < N ? bias[i] : 0.f;
    s.plnw[i] = i < N ? lnw[i] : 0.f;
    s.plnb[i] = i < N ? lnb[i] : 0.f;
  }
  const uint32_t tmem = tc_mainloop(s, tid, row < M, nchunks, [&](int c) {
    return TcChunk{X + row * ldx + c * TC_KC, Kred - c * TC_KC, tiles + (int64_t)c * (2 * NT * TC_KC)};
  });

  // ---- epilogue: thread = row.  z = acc + b, a = act(z), LayerNorm over the N valid columns.
  // Three passes over the accumulator row in TMEM: sum, centred sum of squares (the exact two-pass LayerNorm
  // statistics, in the same summation order as the FP32 SIMT kernel), then Z and Y of a 64-column half tile are
  // formed together and transposed through the (now idle) operand stages -- two XOR-swizzled half tiles, conflict
  // free for the row-per-thread writes and the row-per-warp reads -- into full-row coalesced global stores.
  // Parameters are read from shared memory as broadcast float4 (one LDS per 4 columns: the LSU / shared pipe, not
  // the tensor pipe, is what this kernel saturates -- profiles/ncu_bigm_r01_summary.txt).
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  const float inv_n = 1.f / (float)N;
  float sum = 0.f;
  for (int c0 = 0; c0 < N; c0 += 32) {
    float v[32];
    um::tmem_ld32(trow + c0, v);
#pragma unroll
    for (int j4 = 0; j4 < 32; j4 += 4) {
      if (c0 + j4 < N) {  // N is a multiple of 4
        const float4 b4 = *reinterpret_cast<const float4*>(&s.pbias[c0 + j4]);
        sum += act_fwd<ACT>(v[j4] + b4.x);
        sum += act_fwd<ACT>(v[j4 + 1] + b4.y);
        sum += act_fwd<ACT>(v[j4 + 2] + b4.z);
        sum += act_fwd<ACT>(v[j4 + 3] + b4.w);
      }
    }
  }
  const float mean = sum * inv_n;
  float sq = 0.f;
  for (int c0 = 0; c0 < N; c0 += 32) {
    float v[32];
    um::tmem_ld32(trow + c0, v);
#pragma unroll
    for (int j4 = 0; j4 < 32; j4 += 4) {
      if (c0 + j4 < N) {
        const float4 b4 = *reinterpret_cast<const float4*>(&s.pbias[c0 + j4]);
        float d;
        d = act_fwd<ACT>(v[j4] + b4.x) - mean; sq = fmaf(d, d, sq);
        d = act_fwd<ACT>(v[j4 + 1] + b4.y) - mean; sq = fmaf(d, d, sq);
        d = act_fwd<ACT>(v[j4 + 2] + b4.z) - mean; sq = fmaf(d, d, sq);
        d = act_fwd<ACT>(v[j4 + 3] + b4.w) - mean; sq = fmaf(d, d, sq);
      }
    }
  }
  const float rstd = rsqrtf(sq * inv_n + 1e-5f);
  constexpr int NH = NT >= 64 ? 2 : 1;              // column halves
  constexpr int HC = NT / NH;                       // columns per half
  constexpr int CPRH = HC / 4;                      // 16-byte chunks per half-tile row
  constexpr bool kViaSmem = (size_t)2 * TC_BM * HC * 4 <= sizeof(s.a) + sizeof(s.b);
  float4* zt = reinterpret_cast<float4*>(&s.a[0][0][0]);
  float4* yt = zt + TC_BM * CPRH;
  const int nvalid = (int)(M - row0 < TC_BM ? M - row0 : TC_BM);
  const int sw = tid & (CPRH - 1);
#pragma unroll 1
  for (int h = 0; h < NH; ++h) {
    for (int c0 = h * HC; c0 < (h + 1) * HC && c0 < N; c0 += 32) {
      float v[32];
      um::tmem_ld32(trow + c0, v);
#pragma unroll
      for (int j4 = 0; j4 < 32; j4 += 4) {
        if (c0 + j4 < N && c0 + j4 < (h + 1) * HC) {
          const float4 b4 = *reinterpret_cast<const float4*>(&s.pbias[c0 + j4]);
          const float4 g4 = *reinterpret_cast<const float4*>(&s.plnw[c0 + j4]);
          const float4 e4 = *reinterpret_cast<const float4*>(&s.plnb[c0 + j4]);
          const float4 z4 = make_float4(v[j4] + b4.x, v[j4 + 1] + b4.y, v[j4 + 2] + b4.z, v[j4 + 3] + b4.w);
          const float4 y4 = make_float4((act_fwd<ACT>(z4.x) - mean) * rstd * g4.x + e4.x, (act_fwd<ACT>(z4.y) - mean) * rstd * g4.y + e4.y,
                                        (act_fwd<ACT>(z4.z) - mean) * rstd * g4.z + e4.z, (act_fwd<ACT>(z4.w) - mean) * rstd * g4.w + e4.w);
          if (kViaSmem) {
            const int ch = (c0 - h * HC + j4) >> 2;
            if (Z != nullptr) zt[tid * CPRH + (ch ^ sw)] = z4;
            yt[tid * CPRH + (ch ^ sw)] = y4;
          } else if (row < M) {
            if (Z != nullptr) *reinterpret_cast<float4*>(Z + row * N + c0 + j4) = z4;
            *reinterpret_cast<float4*>(Y + row * N + c0 + j4) = y4;
          }
        }
      }
    }
    if (kViaSmem) {
      __syncthreads();
      for (int i = tid; i < TC_BM * CPRH; i += 128) {
        const int r = i / CPRH, lc = i % CPRH;
        const int col = h * HC + lc * 4;
        if (r < nvalid && col < N) {
          const int slot = r * CPRH + (lc ^ (r & (CPRH - 1)));
          if (Z != nullptr) *reinterpret_cast<float4*>(Z + (row0 + r) * N + col) = zt[slot];
          *reinterpret_cast<float4*>(Y + (row0 + r) * N + col) = yt[slot];
        }
      }
      __syncthreads();
    }
  }
  if (stats != nullptr && row < M) { stats[row * 2] = mean; stats[row * 2 + 1] = rstd; }

  um::tc_fence_before();
  __syncthreads();
  if (warp == 0) um::tmem_dealloc(tmem, NT);
}

template <int NT>
static int launch_tc_fwd_nt(int act, const float* X, int ldx, const float* tiles, int nchunks, const float* bias,
                            const float* lnw, const float* lnb, float* Z, float* Y, float* stats, int64_t M, int N,
                            int Kred, cudaStream_t st) {
  const size_t smem = sizeof(TcSmem<NT>) + 1024;
  dim3 grid((unsigned)ceil_div64(M, TC_BM));
#define HB_TC_CASE(A)                                                                                       \
  case A: {                                                                                                 \
    auto kern = tc_linear_ln_fwd_kernel<NT, A>;                                                             \
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                     \
    kern<<<grid, 128, smem, st>>>(X, ldx, tiles, nchunks, bias, lnw, lnb, Z, Y, stats, M, N, Kred);         \
  } break;
  switch (act) {
    HB_TC_CASE(HB_ACT_RELU) HB_TC_CASE(HB_ACT_TANH) HB_TC_CASE(HB_ACT_SIGMOID) HB_TC_CASE(HB_ACT_LEAKY_RELU)
    HB_TC_CASE(HB_ACT_SELU) HB_TC_CASE(HB_ACT_HARDSWISH) HB_TC_CASE(HB_ACT_IDENTITY)
    default: set_error("activation %d", act); return HB_ERR_UNSUPPORTED;
  }
#undef HB_TC_CASE
  HB_LAUNCH_DONE(st, shape_label("tc_linear_ln_fwd_3xtf32", M, N, Kred));
  return HB_OK;
}

int tc_nt_of(int n) { return n <= 32 ? 32 : n <= 64 ? 64 : n <= 128 ? 128 : 256; }

int launch_tc_linear_ln_fwd(int act, const float* X, int ldx, const float* tiles, int nchunks,
                            const float* bias, const float* lnw, const float* lnb, float* Z, float* Y, float* stats,
                            int64_t M, int N, int Kred, cudaStream_t st) {
  if (M <= 0) return HB_OK;
  const int nt = tc_nt_of(N);
#define HB_TC_NT(NTV)                                                                                              \
  case NTV:                                                                                                        \
    return launch_tc_fwd_nt<NTV>(act, X, ldx, tiles, nchunks, bias, lnw, lnb, Z, Y, stats, M, N, Kred, st);
  switch (nt) { HB_TC_NT(32) HB_TC_NT(64) HB_TC_NT(128) HB_TC_NT(256) }
#undef HB_TC_NT
  return HB_ERR_UNSUPPORTED;
}

}  // namespace hb

// =====================================================================================================
// Backward kernels on tcgen05
// =====================================================================================================
namespace hb {

// slots of the split gradient buffer = CTAs of the dW kernel: three per SM (its 64 KB operand stage allows three)
__host__ __device__ constexpr int tc_dw_splits_c() { return 444; }

// Column sums over the 32 lanes of a warp for 32 per-lane values: lane l ends with sum_lanes v[l].
// Reduce-scatter butterfly: 31 shuffles instead of 32 full reductions.
__device__ __forceinline__ float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int j = 0; j < off; ++j) {
      const float send = up ? v[j] : v[j + off];
      const float keep = up ? v[j + off] : v[j];
      v[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

// ---- dYp = dZ [M,N] W [N,Np] on tensor cores, then LN-backward + act' of the previous block (thread = row)
template <int NT, int ACT>
__global__ void __launch_bounds__(128, 1) tc_dx_ln_bwd_kernel(const float* __restrict__ dZ, int N,
                                                              const float* __restrict__ tiles, int nchunks,
                                                              const float* __restrict__ Zp, const float* __restrict__ stats_p,
                                                              const float* __restrict__ lnw_p, float* __restrict__ dZp,
                                                              float* __restrict__ g_lnw_p, float* __restrict__ g_lnb_p,
                                                              int64_t M, int Np, int64_t part_delta, int64_t part_stride) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  TcSmem<NT>& s = *reinterpret_cast<TcSmem<NT>*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t row0 = (int64_t)blockIdx.x * TC_BM;
  const int64_t row = row0 + tid;
  const uint32_t tmem = tc_mainloop(s, tid, row < M, nchunks, [&](int c) {
    return TcChunk{dZ + row * N + c * TC_KC, N - c * TC_KC, tiles + (int64_t)c * (2 * NT * TC_KC)};
  });

  // ---- epilogue.  Parameters / column sums live in the small shared arrays; the Zp tile is staged through the (now
  // idle) operand stage with coalesced loads and an XOR chunk swizzle, transformed in place into dZp by its row's
  // thread, and written out with coalesced stores (NT <= 128; wider tiles use direct row accesses).
  float* colsum = s.pbias;  // [2][NT] (pbias, plnw are contiguous)
  for (int i = tid; i < NT; i += 128) { s.pbias[i] = 0.f; s.plnw[i] = 0.f; s.plnb[i] = i < Np ? lnw_p[i] : 0.f; }
  constexpr int CPR = NT / 4;
  constexpr bool kViaSmem = (size_t)TC_BM * NT * 4 <= sizeof(s.a) + sizeof(s.b);
  float4* tile = reinterpret_cast<float4*>(&s.a[0][0][0]);
  const int nvalid = (int)(M - row0 < TC_BM ? M - row0 : TC_BM);
  if (kViaSmem) {
    for (int i = tid; i < TC_BM * CPR; i += 128) {
      const int r = i / CPR, lc = i % CPR;
      float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < nvalid && lc * 4 < Np) z = *reinterpret_cast<const float4*>(Zp + (row0 + r) * Np + lc * 4);
      tile[r * CPR + (lc ^ (r & (CPR - 1) & 31))] = z;
    }
  }
  __syncthreads();
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  const bool rok = row < M;
  const int sw = tid & (CPR - 1) & 31;
  float mu = 0.f, rstd = 0.f;
  if (rok) { mu = stats_p[row * 2]; rstd = stats_p[row * 2 + 1]; }
  const float inv_n = 1.f / (float)Np;
  float s1 = 0.f, s2 = 0.f;
  for (int c0 = 0; c0 < Np; c0 += 32) {
    float v[32], cg[32], cb[32];
    um::tmem_ld32(trow + c0, v);
#pragma unroll
    for (int j4 = 0; j4 < 32; j4 += 4) {
      float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      const bool ok = rok && c0 + j4 < Np;
      if (kViaSmem) { if (c0 + j4 < NT) z = tile[tid * CPR + ((((c0 + j4) >> 2)) ^ sw)]; }
      else if (ok) z = *reinterpret_cast<const float4*>(Zp + row * Np + c0 + j4);
      const float zz[4] = {z.x, z.y, z.z, z.w};
      const float4 w4 = *reinterpret_cast<const float4*>(&s.plnb[c0 + j4 < NT ? c0 + j4 : 0]);
      const float ww[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float dy = ok ? v[j4 + q] : 0.f;
        const float x = ok ? (act_fwd<ACT>(zz[q]) - mu) * rstd : 0.f;
        const float g = ok ? dy * ww[q] : 0.f;
        cg[j4 + q] = dy * x;
        cb[j4 + q] = dy;
        s1 += g;
        s2 = fmaf(g, x, s2);
      }
    }
    const float a = warp_colsum32(cg, lane), b = warp_colsum32(cb, lane);
    if (c0 + lane < Np) { atomicAdd(&colsum[c0 + lane], a); atomicAdd(&colsum[NT + c0 + lane], b); }
  }
  const float m1 = s1 * inv_n, m2 = s2 * inv_n;
  for (int c0 = 0; c0 < Np; c0 += 32) {
    float v[32];
    um::tmem_ld32(trow + c0, v);
#pragma unroll
    for (int j4 = 0; j4 < 32; j4 += 4) {
      if (c0 + j4 < Np) {
        float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        const int slot = tid * CPR + (((c0 + j4) >> 2) ^ sw);
        if (kViaSmem) z = tile[slot];
        else if (rok) z = *reinterpret_cast<const float4*>(Zp + row * Np + c0 + j4);
        const float zz[4] = {z.x, z.y, z.z, z.w};
        const float4 w4 = *reinterpret_cast<const float4*>(&s.plnb[c0 + j4]);
        const float ww[4] = {w4.x, w4.y, w4.z, w4.w};
        float o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float x = (act_fwd<ACT>(zz[q]) - mu) * rstd;
          const float g = v[j4 + q] * ww[q];
          o[q] = rstd * (g - m1 - x * m2) * act_bwd<ACT>(zz[q]);
        }
        const float4 o4 = make_float4(o[0], o[1], o[2], o[3]);
        if (kViaSmem) tile[slot] = o4;
        else if (rok) *reinterpret_cast<float4*>(dZp + row * Np + c0 + j4) = o4;
      }
    }
  }
  if (kViaSmem) {
    __syncthreads();
    for (int i = tid; i < TC_BM * CPR; i += 128) {
      const int r = i / CPR, lc = i % CPR;
      if (r < nvalid && lc * 4 < Np)
        *reinterpret_cast<float4*>(dZp + (row0 + r) * Np + lc * 4) = tile[r * CPR + (lc ^ (r & (CPR - 1) & 31))];
    }
  }
  __syncthreads();
  {
    const int64_t slot = part_stride ? part_delta + (int64_t)(blockIdx.x % (unsigned)tc_dw_splits_c()) * part_stride : 0;
    for (int n = tid; n < Np; n += 128) { acc_out(g_lnw_p + n, colsum[n], slot); acc_out(g_lnb_p + n, colsum[NT + n], slot); }
  }
  um::tc_fence_before();
  __syncthreads();
  if (warp == 0) um::tmem_dealloc(tmem, NT);
}

template <int NT>
static int launch_tc_dx_nt(int act, const float* dZ, int N, const float* tiles, int nchunks, const float* Zp,
                           const float* stats_p, const float* lnw_p, float* dZp, float* g_lnw_p, float* g_lnb_p,
                           int64_t M, int Np, int64_t part_delta, int64_t part_stride, cudaStream_t st) {
  const size_t smem = sizeof(TcSmem<NT>) + 1024;
  dim3 grid((unsigned)ceil_div64(M, TC_BM));
#define HB_TC_CASE(A)                                                                                       \
  case A: {                                                                                                 \
    auto kern = tc_dx_ln_bwd_kernel<NT, A>;                                                                 \
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                     \
    kern<<<grid, 128, smem, st>>>(dZ, N, tiles, nchunks, Zp, stats_p, lnw_p, dZp, g_lnw_p, g_lnb_p, M, Np, part_delta, part_stride); \
  } break;
  switch (act) {
    HB_TC_CASE(HB_ACT_RELU) HB_TC_CASE(HB_ACT_TANH) HB_TC_CASE(HB_ACT_SIGMOID) HB_TC_CASE(HB_ACT_LEAKY_RELU)
    HB_TC_CASE(HB_ACT_SELU) HB_TC_CASE(HB_ACT_HARDSWISH) HB_TC_CASE(HB_ACT_IDENTITY)
    default: set_error("activation %d", act); return HB_ERR_UNSUPPORTED;
  }
#undef HB_TC_CASE
  HB_LAUNCH_DONE(st, shape_label("tc_dx_ln_bwd_3xtf32", M, Np, N));
  return HB_OK;
}

int launch_tc_dx_ln_bwd(int act, const float* dZ, int N, const float* tiles, int nchunks, const float* Zp,
                        const float* stats_p, const float* lnw_p, float* dZp, float* g_lnw_p, float* g_lnb_p, int64_t M,
                        int Np, int64_t part_delta, int64_t part_stride, cudaStream_t st) {
  if (M <= 0) return HB_OK;
#define HB_TC_NT(NTV)                                                                                                   \
  case NTV:                                                                                                             \
    return launch_tc_dx_nt<NTV>(act, dZ, N, tiles, nchunks, Zp, stats_p, lnw_p, dZp, g_lnw_p, g_lnb_p, M, Np, part_delta, part_stride, st);
  switch (tc_nt_of(Np)) { HB_TC_NT(32) HB_TC_NT(64) HB_TC_NT(128) HB_TC_NT(256) }
#undef HB_TC_NT
  return HB_ERR_UNSUPPORTED;
}

// ---- Tangent of one Linear -> act -> LayerNorm block on tensor cores, for the trust-region Fisher-vector product
// (trpo.cu; the default tangent block, hb_set_trpo_jvp_impl(1)).
//   acc = Xd W^T + X Wd^T  as ONE accumulation over 2 x nchunks operand chunks (phase 0: A = Xd, B = the forward
//   weight images; phase 1: A = X, B = images of the tangent weights packed per product by pack_umma_tiles), then
//   ad = act'(Z) (acc + bd);  xh = (act(Z) - mu) rstd;  yd = gd xh + betad + g rstd (ad - mean(ad) - xh mean(xh ad)).
// Z-tile staging is that of tc_dx_ln_bwd_kernel (thread = row in the epilogue); pbias <- bd, plnw <- g,
// plnb <- gd, betad is read from global memory (broadcast).  Xd == nullptr (first layer: the normalised observations
// carry no tangent) runs phase 1 only.
template <int NT, int ACT>
__global__ void __launch_bounds__(128, 1) tc_jvp_linear_ln_kernel(const float* __restrict__ X, int ldx,
                                                                  const float* __restrict__ Xd,
                                                                  const float* __restrict__ tiles,
                                                                  const float* __restrict__ tiles_d, int nchunks,
                                                                  const float* __restrict__ bd, const float* __restrict__ lnw,
                                                                  const float* __restrict__ lnwd, const float* __restrict__ lnbd,
                                                                  const float* __restrict__ Zp, const float* __restrict__ stats_p,
                                                                  float* __restrict__ Yd, int64_t M, int Np, int Kred) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  TcSmem<NT>& s = *reinterpret_cast<TcSmem<NT>*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int64_t row0 = (int64_t)blockIdx.x * TC_BM;
  const int64_t row = row0 + tid;
  for (int i = tid; i < NT; i += 128) {
    s.pbias[i] = i < Np ? bd[i] : 0.f;
    s.plnw[i] = i < Np ? lnw[i] : 0.f;
    s.plnb[i] = i < Np ? lnwd[i] : 0.f;
  }
  const int first = Xd != nullptr ? 0 : nchunks;   // chunk counter runs over [first, 2 nchunks)
  const uint32_t tmem = tc_mainloop(s, tid, row < M, 2 * nchunks - first, [&](int i) {
    const int cc = first + i;
    const bool tangent_w = cc >= nchunks;          // phase 1: A = X, B = tangent weight images
    const int c = tangent_w ? cc - nchunks : cc;
    return TcChunk{(tangent_w ? X : Xd) + row * ldx + c * TC_KC, Kred - c * TC_KC,
                   (tangent_w ? tiles_d : tiles) + (int64_t)c * (2 * NT * TC_KC)};
  });

  // ---- epilogue (thread = row): Z tile staged through the idle operand stage, transformed in place into yd
  constexpr int CPR = NT / 4;
  constexpr bool kViaSmem = (size_t)TC_BM * NT * 4 <= sizeof(s.a) + sizeof(s.b);
  float4* tile = reinterpret_cast<float4*>(&s.a[0][0][0]);
  const int nvalid = (int)(M - row0 < TC_BM ? M - row0 : TC_BM);
  if (kViaSmem) {
    for (int i = tid; i < TC_BM * CPR; i += 128) {
      const int r = i / CPR, lc = i % CPR;
      float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < nvalid && lc * 4 < Np) z = *reinterpret_cast<const float4*>(Zp + (row0 + r) * Np + lc * 4);
      tile[r * CPR + (lc ^ (r & (CPR - 1) & 31))] = z;
    }
  }
  __syncthreads();
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  const bool rok = row < M;
  const int sw = tid & (CPR - 1) & 31;
  float mu = 0.f, rstd = 0.f;
  if (rok) { mu = stats_p[row * 2]; rstd = stats_p[row * 2 + 1]; }
  const float inv_n = 1.f / (float)Np;
  float s1 = 0.f, s2 = 0.f;
  for (int c0 = 0; c0 < Np; c0 += 32) {
    float v[32];
    um::tmem_ld32(trow + c0, v);
#pragma unroll
    for (int j4 = 0; j4 < 32; j4 += 4) {
      if (c0 + j4 < Np) {
        float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        if (kViaSmem) z = tile[tid * CPR + (((c0 + j4) >> 2) ^ sw)];
        else if (rok) z = *reinterpret_cast<const float4*>(Zp + row * Np + c0 + j4);
        const float zz[4] = {z.x, z.y, z.z, z.w};
        const float4 b4 = *reinterpret_cast<const float4*>(&s.pbias[c0 + j4]);
        const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float ad = rok ? act_bwd<ACT>(zz[q]) * (v[j4 + q] + bb[q]) : 0.f;
          const float x = rok ? (act_fwd<ACT>(zz[q]) - mu) * rstd : 0.f;
          s1 += ad;
          s2 = fmaf(ad, x, s2);
        }
      }
    }
  }
  const float m1 = s1 * inv_n, m2 = s2 * inv_n;
  for (int c0 = 0; c0 < Np; c0 += 32) {
    float v[32];
    um::tmem_ld32(trow + c0, v);
#pragma unroll
    for (int j4 = 0; j4 < 32; j4 += 4) {
      if (c0 + j4 < Np) {
        float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        const int slot = tid * CPR + (((c0 + j4) >> 2) ^ sw);
        if (kViaSmem) z = tile[slot];
        else if (rok) z = *reinterpret_cast<const float4*>(Zp + row * Np + c0 + j4);
        const float zz[4] = {z.x, z.y, z.z, z.w};
        const float4 b4 = *reinterpret_cast<const float4*>(&s.pbias[c0 + j4]);
        const float4 g4 = *reinterpret_cast<const float4*>(&s.plnw[c0 + j4]);
        const float4 d4 = *reinterpret_cast<const float4*>(&s.plnb[c0 + j4]);
        const float4 e4 = __ldg(reinterpret_cast<const float4*>(lnbd + c0 + j4));
        const float bb[4] = {b4.x, b4.y, b4.z, b4.w}, gg[4] = {g4.x, g4.y, g4.z, g4.w};
        const float dd[4] = {d4.x, d4.y, d4.z, d4.w}, ee[4] = {e4.x, e4.y, e4.z, e4.w};
        float o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float ad = act_bwd<ACT>(zz[q]) * (v[j4 + q] + bb[q]);
          const float x = (act_fwd<ACT>(zz[q]) - mu) * rstd;
          o[q] = dd[q] * x + ee[q] + gg[q] * rstd * (ad - m1 - x * m2);
        }
        const float4 o4 = make_float4(o[0], o[1], o[2], o[3]);
        if (kViaSmem) tile[slot] = o4;
        else if (rok) *reinterpret_cast<float4*>(Yd + row * Np + c0 + j4) = o4;
      }
    }
  }
  if (kViaSmem) {
    __syncthreads();
    for (int i = tid; i < TC_BM * CPR; i += 128) {
      const int r = i / CPR, lc = i % CPR;
      if (r < nvalid && lc * 4 < Np)
        *reinterpret_cast<float4*>(Yd + (row0 + r) * Np + lc * 4) = tile[r * CPR + (lc ^ (r & (CPR - 1) & 31))];
    }
  }
  um::tc_fence_before();
  __syncthreads();
  if (warp == 0) um::tmem_dealloc(tmem, NT);
}

template <int NT>
static int launch_tc_jvp_nt(int act, const float* X, int ldx, const float* Xd, const float* tiles, const float* tiles_d,
                            int nchunks, const float* bd, const float* lnw, const float* lnwd, const float* lnbd,
                            const float* Z, const float* stats, float* Yd, int64_t M, int N, int Kred, cudaStream_t st) {
  const size_t smem = sizeof(TcSmem<NT>) + 1024;
  dim3 grid((unsigned)ceil_div64(M, TC_BM));
#define HB_TC_CASE(A)                                                                                       \
  case A: {                                                                                                 \
    auto kern = tc_jvp_linear_ln_kernel<NT, A>;                                                             \
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);                     \
    kern<<<grid, 128, smem, st>>>(X, ldx, Xd, tiles, tiles_d, nchunks, bd, lnw, lnwd, lnbd, Z, stats, Yd, M, N, Kred); \
  } break;
  switch (act) {
    HB_TC_CASE(HB_ACT_RELU) HB_TC_CASE(HB_ACT_TANH) HB_TC_CASE(HB_ACT_SIGMOID) HB_TC_CASE(HB_ACT_LEAKY_RELU)
    HB_TC_CASE(HB_ACT_SELU) HB_TC_CASE(HB_ACT_HARDSWISH) HB_TC_CASE(HB_ACT_IDENTITY)
    default: set_error("activation %d", act); return HB_ERR_UNSUPPORTED;
  }
#undef HB_TC_CASE
  HB_LAUNCH_DONE(st, shape_label("tc_jvp_linear_ln_3xtf32", M, N, Kred));
  return HB_OK;
}

int launch_tc_jvp_linear_ln(int act, const float* X, int ldx, const float* Xd, const float* tiles,
                            const float* tiles_d, int nchunks, const float* bd, const float* lnw, const float* lnwd,
                            const float* lnbd, const float* Z, const float* stats, float* Yd, int64_t M, int N, int Kred,
                            cudaStream_t st) {
  if (M <= 0) return HB_OK;
#define HB_TC_NT(NTV)                                                                                                   \
  case NTV:                                                                                                             \
    return launch_tc_jvp_nt<NTV>(act, X, ldx, Xd, tiles, tiles_d, nchunks, bd, lnw, lnwd, lnbd, Z, stats, Yd, M, N, Kred, st);
  switch (tc_nt_of(N)) { HB_TC_NT(32) HB_TC_NT(64) HB_TC_NT(128) HB_TC_NT(256) }
#undef HB_TC_NT
  return HB_ERR_UNSUPPORTED;
}

// ---- dW[n][k] += sum_r dZ[r][n] X[r][k].  The row index r is the MMA K dimension, so both operands are staged
// TRANSPOSED into the same K-major image the forward kernels use:  image(f, r) = [f/8][r/4][f%8][r%4].
// Thread t owns feature t: it reads 4 consecutive rows of its column with scalar loads (coalesced across the
// warp: 32 neighbouring features of one row = 128 B) and writes one 16-byte slot (conflict-free: 8 neighbouring
// features fill 128 contiguous bytes).  One CTA: 128 dZ features (grid.y) x all NTK X features over a slice of rows
// (grid.x); fp32 accumulator in TMEM; epilogue: thread = dZ feature, atomicAdd of its dW row; db from the staging sums.
template <int NTK>
struct TcDwSmem {
  float a[TC_STAGES][2][TC_KC * 128];   // [stage][hi/lo] dZ^T chunk image (128 features x 32 rows)
  float b[TC_STAGES][2][TC_KC * NTK];   // [stage][hi/lo] X^T chunk image (NTK features x 32 rows)
  uint64_t empty[TC_STAGES];
  uint64_t done;
  uint32_t tmem_base;
};

template <int NTK>
__global__ void __launch_bounds__(128, 1) tc_dw_accum_kernel(const float* __restrict__ dZ, int N,
                                                             const float* __restrict__ X, int ldx, int K,
                                                             float* __restrict__ dW, float* __restrict__ db, int64_t M,
                                                             int64_t rows_per_cta, int64_t part_stride) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  TcDwSmem<NTK>& s = *reinterpret_cast<TcDwSmem<NTK>*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5;
  const int n0 = blockIdx.y * 128;
  const int k0 = blockIdx.z * NTK;   // X feature block (input widths > 256, e.g. 393-wide observations)
  const int64_t m0 = (int64_t)blockIdx.x * rows_per_cta;
  const int64_t m1 = m0 + rows_per_cta < M ? m0 + rows_per_cta : M;
  if (tid == 0) {
    for (int i = 0; i < TC_STAGES; ++i) um::mbar_init(&s.empty[i], 1);
    um::mbar_init(&s.done, 1);
    um::fence_mbarrier_init();
  }
  if (warp == 0) um::tmem_alloc(&s.tmem_base, NTK);
  um::tc_fence_before();
  __syncthreads();
  um::tc_fence_after();
  const uint32_t tmem = s.tmem_base;
  constexpr uint32_t idesc = um::idesc_tf32(NTK);
  const int nchunks = (int)((m1 - m0 + TC_KC - 1) / TC_KC);
  uint32_t ph_empty[2] = {0, 0};
  float bsum = 0.f;
  const int fa = n0 + tid;                                   // this thread's dZ feature
  const int slot = ((tid >> 3) * 8) * 32 + (tid & 7) * 4;    // floats; + kc*32 per 4-row group
  // Register double buffering: the global loads of chunk c + 1 are issued right after chunk c went to shared memory,
  // so their latency overlaps the fence / barrier / MMAs of chunk c instead of adding to every chunk's critic path
  // (the single operand stage keeps three CTAs per SM).
  constexpr int NB = (NTK + 127) / 128;    // X features per thread
  float va[TC_KC], vb[NB][TC_KC];
  auto load_chunk = [&](int c) {
    const int64_t r0 = m0 + (int64_t)c * TC_KC;
#pragma unroll
    for (int q = 0; q < TC_KC; ++q) {
      const int64_t r = r0 + q;
      va[q] = (r < m1 && fa < N) ? dZ[r * N + fa] : 0.f;
    }
#pragma unroll
    for (int fb = 0; fb < NB; ++fb) {
      const int f = fb * 128 + tid;
#pragma unroll
      for (int q = 0; q < TC_KC; ++q) {
        const int64_t r = r0 + q;
        vb[fb][q] = (f < NTK && r < m1 && k0 + f < ldx) ? X[r * ldx + k0 + f] : 0.f;
      }
    }
  };
  if (nchunks > 0) load_chunk(0);
  for (int c = 0; c < nchunks; ++c) {
    const int st = c % TC_STAGES;
    if (c >= TC_STAGES) { um::mbar_wait(&s.empty[st], ph_empty[st]); ph_empty[st] ^= 1; }
#pragma unroll
    for (int kc = 0; kc < 8; ++kc) {
      const float* v = va + kc * 4;
      bsum += (v[0] + v[1]) + (v[2] + v[3]);
      const float4 h = make_float4(tf32_hi(v[0]), tf32_hi(v[1]), tf32_hi(v[2]), tf32_hi(v[3]));
      *reinterpret_cast<float4*>(&s.a[st][0][slot + kc * 32]) = h;
      *reinterpret_cast<float4*>(&s.a[st][1][slot + kc * 32]) = make_float4(tf32_lo(v[0], h.x), tf32_lo(v[1], h.y), tf32_lo(v[2], h.z), tf32_lo(v[3], h.w));
    }
#pragma unroll
    for (int fb = 0; fb < NB; ++fb) {
      const int f = fb * 128 + tid;
      if (f < NTK) {
        const int bslot = ((f >> 3) * 8) * 32 + (f & 7) * 4;
#pragma unroll
        for (int kc = 0; kc < 8; ++kc) {
          const float* v = vb[fb] + kc * 4;
          const float4 h = make_float4(tf32_hi(v[0]), tf32_hi(v[1]), tf32_hi(v[2]), tf32_hi(v[3]));
          *reinterpret_cast<float4*>(&s.b[st][0][bslot + kc * 32]) = h;
          *reinterpret_cast<float4*>(&s.b[st][1][bslot + kc * 32]) = make_float4(tf32_lo(v[0], h.x), tf32_lo(v[1], h.y), tf32_lo(v[2], h.z), tf32_lo(v[3], h.w));
        }
      }
    }
    if (c + 1 < nchunks) load_chunk(c + 1);
    um::fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      um::tc_fence_after();
      const uint32_t a_hi = um::smem_u32(s.a[st][0]), a_lo = um::smem_u32(s.a[st][1]);
      const uint32_t b_hi = um::smem_u32(s.b[st][0]), b_lo = um::smem_u32(s.b[st][1]);
#pragma unroll
      for (int j = 0; j < TC_KC / 8; ++j) {
        const uint32_t off = j * 256;
        const uint64_t dah = um::desc(a_hi + off, 128, 1024), dbh = um::desc(b_hi + off, 128, 1024);
        um::mma_tf32(tmem, dah, dbh, idesc, (c | j) != 0);
        const uint64_t dal = um::desc(a_lo + off, 128, 1024), dbl = um::desc(b_lo + off, 128, 1024);
        um::mma_tf32(tmem, dal, dbh, idesc, 1);
        um::mma_tf32(tmem, dah, dbl, idesc, 1);
      }
      um::commit(&s.empty[st]);
      if (c == nchunks - 1) um::commit(&s.done);
    }
  }
  if (nchunks > 0) {
    um::mbar_wait(&s.done, 0);
    um::tc_fence_after();
    const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
    // part_stride != 0: this CTA owns slot blockIdx.x of a split buffer [splits][params] -> plain read-modify-write
    // (deterministic, no atomics; summed into the gradient once per call by dw_reduce_kernel).  Else: atomics into dW.
    float* dst = dW + (int64_t)blockIdx.x * part_stride + (int64_t)fa * K;
    for (int c0 = 0; c0 < NTK && k0 + c0 < K; c0 += 32) {
      float v[32];
      um::tmem_ld32(trow + c0, v);
      if (fa < N) {
        if (part_stride != 0 && (K & 3) == 0) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            if (k0 + c0 + j < K) {
              float4* q = reinterpret_cast<float4*>(dst + k0 + c0 + j);
              float4 o = *q;
              o.x += v[j]; o.y += v[j + 1]; o.z += v[j + 2]; o.w += v[j + 3];
              *q = o;
            }
          }
        } else if (part_stride != 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (k0 + c0 + j < K) dst[k0 + c0 + j] += v[j];
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (k0 + c0 + j < K) atomicAdd(dst + k0 + c0 + j, v[j]);
        }
      }
    }
    if (db != nullptr && fa < N && blockIdx.z == 0) atomicAdd(db + fa, bsum);
  }
  um::tc_fence_before();
  __syncthreads();
  if (warp == 0) um::tmem_dealloc(tmem, NTK);
}

constexpr int TC_DW_SPLITS = tc_dw_splits_c();

__global__ void dw_reduce_kernel(float* __restrict__ grad, const float* __restrict__ part, int splits, int total) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  float acc = 0.f;
#pragma unroll 8
  for (int s = 0; s < splits; ++s) acc += part[(int64_t)s * total + i];
  grad[i] += acc;
}

int tc_dw_splits() { return TC_DW_SPLITS; }

int launch_dw_reduce(float* grad, const float* part, int total, cudaStream_t st) {
  dw_reduce_kernel<<<(total + 127) / 128, 128, 0, st>>>(grad, part, TC_DW_SPLITS, total);
  HB_LAUNCH_DONE(st, "dw_reduce");
  return HB_OK;
}

template <int NTK>
static int launch_tc_dw_ntk(const float* dZ, int N, const float* X, int ldx, int K, float* dW, float* db,
                            int64_t M, int64_t part_stride, cudaStream_t st) {
  const int nb = (N + 127) / 128, kb = (ldx + NTK - 1) / NTK;
  int64_t splits, rows_per;
  if (part_stride != 0) {
    splits = TC_DW_SPLITS;
    rows_per = (ceil_div64(M, splits) + 31) / 32 * 32;
  } else {
    splits = (3 * 148 + nb * kb - 1) / (nb * kb);
    rows_per = (ceil_div64(M, splits) + 31) / 32 * 32;
    if (rows_per < 128) rows_per = 128;
    splits = ceil_div64(M, rows_per);
  }
  const size_t smem = sizeof(TcDwSmem<NTK>) + 1024;
  dim3 grid((unsigned)splits, nb, kb);
  auto kern = tc_dw_accum_kernel<NTK>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  kern<<<grid, 128, smem, st>>>(dZ, N, X, ldx, K, dW, db, M, rows_per, part_stride);
  HB_LAUNCH_DONE(st, shape_label("tc_dw_accum_3xtf32", M, N, K));
  return HB_OK;
}

int launch_tc_dw_accum(const float* dZ, int N, const float* X, int ldx, int K, float* dW, float* db,
                       int64_t M, int64_t part_stride, cudaStream_t st) {
  if (M <= 0) return HB_OK;
  switch (tc_nt_of(ldx)) {
    case 32: return launch_tc_dw_ntk<32>(dZ, N, X, ldx, K, dW, db, M, part_stride, st);
    case 64: return launch_tc_dw_ntk<64>(dZ, N, X, ldx, K, dW, db, M, part_stride, st);
    case 128: return launch_tc_dw_ntk<128>(dZ, N, X, ldx, K, dW, db, M, part_stride, st);
    default: return launch_tc_dw_ntk<256>(dZ, N, X, ldx, K, dW, db, M, part_stride, st);
  }
}

}  // namespace hb
