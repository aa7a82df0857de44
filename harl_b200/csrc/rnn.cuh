// GRU layer interface (rnn.cu), used by the sequencing code in capi.cu.
#pragma once
#include "common.cuh"

namespace hb {

struct RnnWork {
  float* mrow;      // [M] mask of each batch row (gathered once)
  float* gi[2];     // [M, 3h] input projections of all steps, per layer
  float* hm[2];     // [M, h]  masked previous state = the recurrent GEMM's input at each step
  float* hs[2];     // [M, h]  new state of each step (the layer's output sequence)
  float* gh;        // [B, 3h] per-step scratch
  float* out;       // [M, h]  LayerNorm(hs[top])
  float* stats;     // [2M]
  // gradient mode
  float* gates[2];  // [M, 4h] r, z, n, (W_hn h + b_hn)
  float* dgi;       // [M, 3h]
  float* dgh;       // [M, 3h]
  float* dhm[2];    // [B, h] ping-pong
  float* dtop;      // [M, h] d loss / d hs[top], written by the head kernel (LN backward fused there)
  float* dx[2];     // [M, h] d loss / d (layer input)
};

struct RnnJvpWork {   // tangent pass of the trust-region Fisher-vector product
  float* gid;       // [M, 3h]
  float* ghd;       // [B, 3h]
  float* hmd[2];    // [M, h] tangent of the masked previous state
  float* hsd[2];    // [M, h] tangent of each step's new state
  float* outd;      // [M, h] tangent of LayerNorm(hs[top])
};

int rnn_impl();            // 0 = launch per step, 1 = persistent per-sequence recurrence (default; h = 64 only)
void set_rnn_impl(int v);
size_t rnn_jvp_floats(const PrepLayout& Q, int64_t M);
int carve_rnn_jvp(const PrepLayout& Q, int64_t M, float* p, RnnJvpWork* w);
int rnn_jvp_forward(const PrepLayout& Q, const float* prep, const float* tprep, const float* X, const float* Xd, int64_t S,
                    int64_t B, const RnnWork& w, const RnnJvpWork& jw, cudaStream_t st);
size_t rnn_work_floats(const PrepLayout& Q, int64_t M, int grad);
int carve_rnn(const PrepLayout& Q, int64_t M, int grad, float* p, RnnWork* w);
int launch_linear_plain(const float* X, int ldx, const float* Bm, int ldb, const float* bias, float* Y, int ldy,
                        int64_t M, int N, int Kred, bool accumulate, cudaStream_t st);
int rnn_forward(const PrepLayout& Q, const float* prep, const float* X, int64_t S, int64_t B, const float* h0,
                const float* masks, const int32_t* index, float* h_out, const RnnWork& w, cudaStream_t st);
int rnn_backward(const ParamLayout& P, const PrepLayout& Q, const float* params, const float* X, int64_t S, int64_t B,
                 float* grad, const RnnWork& w, float** dX_out, cudaStream_t st);

}  // namespace hb
