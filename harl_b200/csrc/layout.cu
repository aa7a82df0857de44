// Parameter layout (reference state_dict order), derived-weight preparation, error plumbing.
#include <stdarg.h>

#include <atomic>

#include "common.cuh"

namespace hb {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("%s: CUDA error %d (%s)", what, (int)e, cudaGetErrorString(e));
  return HB_ERR_CUDA;
}

static int add_tensor(hb_net_layout* L, int* cursor, const char* name, int rows, int cols) {
  int off = round_up(*cursor, 4);
  if (L) {
    int i = L->n_tensors++;
    L->offset[i] = off;
    L->rows[i] = rows;
    L->cols[i] = cols;
    strncpy(L->names[i], name, sizeof(L->names[i]) - 1);
    L->names[i][sizeof(L->names[i]) - 1] = 0;
  }
  *cursor = off + rows * cols;
  return off;
}

// Order follows the reference modules' registration order:
// StochasticPolicy (stochastic_policy.py:33-51): base, rnn, act;  MLPBase (mlp.py:55-62):
// feature_norm, mlp.fc.{3l, 3l+2};  RNNLayer (rnn.py:14-21): rnn.rnn.*, rnn.norm;
// DiagGaussian (distributions.py:80-82): fc_mean registered before log_std is assigned, but
// nn.Module yields own parameters (log_std) before sub-modules (fc_mean);  VNet: v_out.
int tc_nt_of(int n);
int launch_pack_umma_jobs(int njobs, const float* const* W, const int* ldn, const int* ldk, const float* const* scale, const int* N,
                          const int* K, const int* NT, const int* nchunks, float* const* dst, cudaStream_t st);

bool fused_shape_ok(const hb_net_desc* d);   // fused_update.cu
int launch_fused_pack(const hb_net_desc* d, const ParamLayout& P, const PrepLayout& Q, const float* params, float* prepared,
                      cudaStream_t st);

static std::atomic<int> g_gemm_impl{1};  // default: tcgen05 with the fp32-accurate 3xTF32 split
int gemm_impl() { return g_gemm_impl.load(std::memory_order_relaxed); }

int make_layouts(const hb_net_desc* d, ParamLayout* pl, PrepLayout* pp, hb_net_layout* out) {
  if (!d) { set_error("net desc is NULL"); return HB_ERR_INVALID; }
  if (d->n_layers < 1 || d->n_layers > HB_MAX_LAYERS) { set_error("n_layers %d outside 1..%d", d->n_layers, HB_MAX_LAYERS); return HB_ERR_UNSUPPORTED; }
  if (d->in_dim < 1) { set_error("in_dim %d", d->in_dim); return HB_ERR_INVALID; }
  for (int l = 0; l < d->n_layers; ++l)
    if (d->hidden[l] < 4 || d->hidden[l] > 256 || d->hidden[l] % 4) { set_error("hidden size %d unsupported (need multiple of 4 in 4..256)", d->hidden[l]); return HB_ERR_UNSUPPORTED; }
  if (d->activation < 0 || d->activation > HB_ACT_IDENTITY) { set_error("activation %d unsupported", d->activation); return HB_ERR_UNSUPPORTED; }
  if (d->head < 0 || d->head > HB_HEAD_VALUE) { set_error("head %d unsupported", d->head); return HB_ERR_UNSUPPORTED; }
  if (d->out_dim < 1 || d->out_dim > 32) { set_error("out_dim %d unsupported (1..32)", d->out_dim); return HB_ERR_UNSUPPORTED; }
  if (d->rnn_layers < 0 || d->rnn_layers > 2) { set_error("rnn_layers %d unsupported", d->rnn_layers); return HB_ERR_UNSUPPORTED; }
  ParamLayout P;
  memset(&P, 0xff, sizeof(P));
  if (out) memset(out, 0, sizeof(*out));
  int cur = 0;
  char nm[64];
  if (d->feature_norm) {
    P.fn_w = add_tensor(out, &cur, "base.feature_norm.weight", 1, d->in_dim);
    P.fn_b = add_tensor(out, &cur, "base.feature_norm.bias", 1, d->in_dim);
  }
  int prev = d->in_dim;
  for (int l = 0; l < d->n_layers; ++l) {
    int h = d->hidden[l];
    snprintf(nm, sizeof nm, "base.mlp.fc.%d.weight", 3 * l); P.w[l] = add_tensor(out, &cur, nm, h, prev);
    snprintf(nm, sizeof nm, "base.mlp.fc.%d.bias", 3 * l);   P.b[l] = add_tensor(out, &cur, nm, 1, h);
    snprintf(nm, sizeof nm, "base.mlp.fc.%d.weight", 3 * l + 2); P.lnw[l] = add_tensor(out, &cur, nm, 1, h);
    snprintf(nm, sizeof nm, "base.mlp.fc.%d.bias", 3 * l + 2);   P.lnb[l] = add_tensor(out, &cur, nm, 1, h);
    prev = h;
  }
  for (int r = 0; r < d->rnn_layers; ++r) {
    snprintf(nm, sizeof nm, "rnn.rnn.weight_ih_l%d", r); P.rnn_wih[r] = add_tensor(out, &cur, nm, 3 * prev, prev);
    snprintf(nm, sizeof nm, "rnn.rnn.weight_hh_l%d", r); P.rnn_whh[r] = add_tensor(out, &cur, nm, 3 * prev, prev);
    snprintf(nm, sizeof nm, "rnn.rnn.bias_ih_l%d", r); P.rnn_bih[r] = add_tensor(out, &cur, nm, 1, 3 * prev);
    snprintf(nm, sizeof nm, "rnn.rnn.bias_hh_l%d", r); P.rnn_bhh[r] = add_tensor(out, &cur, nm, 1, 3 * prev);
  }
  if (d->rnn_layers) {
    P.rnn_lnw = add_tensor(out, &cur, "rnn.norm.weight", 1, prev);
    P.rnn_lnb = add_tensor(out, &cur, "rnn.norm.bias", 1, prev);
  }
  if (d->head == HB_HEAD_DISCRETE) {
    P.hw = add_tensor(out, &cur, "act.action_out.linear.weight", d->out_dim, prev);
    P.hbias = add_tensor(out, &cur, "act.action_out.linear.bias", 1, d->out_dim);
  } else if (d->head == HB_HEAD_BOX) {
    P.log_std = add_tensor(out, &cur, "act.action_out.log_std", 1, d->out_dim);
    P.hw = add_tensor(out, &cur, "act.action_out.fc_mean.weight", d->out_dim, prev);
    P.hbias = add_tensor(out, &cur, "act.action_out.fc_mean.bias", 1, d->out_dim);
  } else {
    P.hw = add_tensor(out, &cur, "v_out.weight", 1, prev);
    P.hbias = add_tensor(out, &cur, "v_out.bias", 1, 1);
  }
  P.total = round_up(cur, 4);

  PrepLayout Q;
  memset(&Q, 0, sizeof(Q));
  Q.n_layers = d->n_layers;
  int c = 0;
  prev = d->in_dim;
  for (int l = 0; l < d->n_layers; ++l) {
    Q.k[l] = prev;
    Q.kpad[l] = round_up(prev, 4);
    Q.n[l] = d->hidden[l];
    Q.wt[l] = c;   c += Q.kpad[l] * Q.n[l];
    Q.bias[l] = c; c += Q.n[l];
    Q.lnw[l] = c;  c += Q.n[l];
    Q.lnb[l] = c;  c += Q.n[l];
    prev = d->hidden[l];
  }
  Q.hw = c;    c += round_up(d->out_dim * prev, 4);
  Q.hbias = c; c += round_up(d->out_dim, 4);
  Q.log_std = c; c += round_up(d->out_dim, 4);
  Q.rnn_layers = d->rnn_layers;
  Q.rh = prev;
  for (int r = 0; r < d->rnn_layers; ++r) {
    Q.rnn_wih_t[r] = c; c += 3 * prev * prev;
    Q.rnn_whh_t[r] = c; c += 3 * prev * prev;
    Q.rnn_bih[r] = c;   c += 3 * prev;
    Q.rnn_bhh[r] = c;   c += 3 * prev;
  }
  if (d->rnn_layers) { Q.rnn_lnw = c; c += prev; Q.rnn_lnb = c; c += prev; }
  for (int l = 0; l < d->n_layers; ++l) {
    Q.tk_nt[l] = tc_nt_of(Q.n[l]);
    Q.tk_chunks[l] = (Q.kpad[l] + 31) / 32;
    Q.tk[l] = c;
    c += Q.tk_chunks[l] * 2 * Q.tk_nt[l] * 32;
  }
  for (int l = 1; l < d->n_layers; ++l) {
    Q.tkt_nt[l] = tc_nt_of(Q.k[l]);
    Q.tkt_chunks[l] = (Q.n[l] + 31) / 32;
    Q.tkt[l] = c;
    c += Q.tkt_chunks[l] * 2 * Q.tkt_nt[l] * 32;
  }
  Q.fz_ok = fused_shape_ok(d) ? 1 : 0;
  if (Q.fz_ok) {
    const int H = d->hidden[0];
    c = round_up(c, 4);                          // TMA bulk copies read the images: 16-byte aligned starts
    Q.fz_k0p = round_up(d->in_dim, 16);
    const int kp[2] = {Q.fz_k0p, H};
    for (int l = 0; l < 2; ++l) {
      Q.fz_chunks[l] = (kp[l] + 31) / 32;
      Q.fz_w[l] = c;    c += H * kp[l];          // 2 images x H x kp halves = H * kp floats
      Q.fz_bias[l] = c; c += H;
    }
    Q.fz_w1b = c;   c += H * H;
    Q.fz_hw = c;    c += 16 * H;                 // 2 images x 16 x H halves
    Q.fz_hbias = c; c += 16;
    Q.fz_scale = c; c += 4;
  }
  Q.total = c;
  if (pl) *pl = P;
  if (pp) *pp = Q;
  if (out) { out->total = P.total; out->prepared_total = Q.total; }
  return HB_OK;
}

__global__ void prepare_kernel(ParamLayout P, PrepLayout Q, int feature_norm, int head, int out_dim,
                               const float* __restrict__ params, float* __restrict__ prep) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Q.total) return;
  for (int l = 0; l < Q.n_layers; ++l) {
    int n = Q.n[l], K = Q.k[l], kp = Q.kpad[l];
    if (i >= Q.wt[l] && i < Q.wt[l] + kp * n) {
      int k = (i - Q.wt[l]) / n, j = (i - Q.wt[l]) % n;
      float v = 0.f;
      if (k < K) {
        v = params[P.w[l] + j * K + k];
        if (l == 0 && feature_norm) v *= params[P.fn_w + k];
      }
      prep[i] = v;
      return;
    }
    if (i >= Q.bias[l] && i < Q.bias[l] + n) {
      int j = i - Q.bias[l];
      float v = params[P.b[l] + j];
      if (l == 0 && feature_norm)
        for (int k = 0; k < K; ++k) v += params[P.w[0] + j * K + k] * params[P.fn_b + k];
      prep[i] = v;
      return;
    }
    if (i >= Q.lnw[l] && i < Q.lnw[l] + n) { prep[i] = params[P.lnw[l] + i - Q.lnw[l]]; return; }
    if (i >= Q.lnb[l] && i < Q.lnb[l] + n) { prep[i] = params[P.lnb[l] + i - Q.lnb[l]]; return; }
  }
  if (i >= Q.tk[0]) return;  // tensor-core operand images are written by pack_umma_jobs
  int h = Q.n[Q.n_layers - 1];
  if (i >= Q.hw && i < Q.hw + out_dim * h) { prep[i] = params[P.hw + i - Q.hw]; return; }
  if (i >= Q.hbias && i < Q.hbias + out_dim) { prep[i] = params[P.hbias + i - Q.hbias]; return; }
  if (head == HB_HEAD_BOX && i >= Q.log_std && i < Q.log_std + out_dim) { prep[i] = params[P.log_std + i - Q.log_std]; return; }
  for (int r = 0; r < Q.rnn_layers; ++r) {
    const int g3 = 3 * h;
    if (i >= Q.rnn_wih_t[r] && i < Q.rnn_wih_t[r] + h * g3) {  // [h][3h] <- W_ih [3h][h]
      int k = (i - Q.rnn_wih_t[r]) / g3, j = (i - Q.rnn_wih_t[r]) % g3;
      prep[i] = params[P.rnn_wih[r] + j * h + k];
      return;
    }
    if (i >= Q.rnn_whh_t[r] && i < Q.rnn_whh_t[r] + h * g3) {
      int k = (i - Q.rnn_whh_t[r]) / g3, j = (i - Q.rnn_whh_t[r]) % g3;
      prep[i] = params[P.rnn_whh[r] + j * h + k];
      return;
    }
    if (i >= Q.rnn_bih[r] && i < Q.rnn_bih[r] + g3) { prep[i] = params[P.rnn_bih[r] + i - Q.rnn_bih[r]]; return; }
    if (i >= Q.rnn_bhh[r] && i < Q.rnn_bhh[r] + g3) { prep[i] = params[P.rnn_bhh[r] + i - Q.rnn_bhh[r]]; return; }
  }
  if (Q.rnn_layers) {
    if (i >= Q.rnn_lnw && i < Q.rnn_lnw + h) { prep[i] = params[P.rnn_lnw + i - Q.rnn_lnw]; return; }
    if (i >= Q.rnn_lnb && i < Q.rnn_lnb + h) { prep[i] = params[P.rnn_lnb + i - Q.rnn_lnb]; return; }
  }
  prep[i] = 0.f;
}

int prepare_launch(const hb_net_desc* d, const float* params, float* prepared, cudaStream_t st) {
  ParamLayout P;
  PrepLayout Q;
  int rc = make_layouts(d, &P, &Q, nullptr);
  if (rc) return rc;
  prepare_kernel<<<(Q.tk[0] + 255) / 256, 256, 0, st>>>(P, Q, d->feature_norm, d->head, d->out_dim, params, prepared);
  HB_LAUNCH_DONE(st,"hb_net_prepare");
  if (gemm_impl() != 0) {  // all tcgen05 operand images of the layer-wise kernels in one launch
    const float* W[2 * HB_MAX_LAYERS]; const float* sc[2 * HB_MAX_LAYERS]; float* dst[2 * HB_MAX_LAYERS];
    int ldn[2 * HB_MAX_LAYERS], ldk[2 * HB_MAX_LAYERS], N[2 * HB_MAX_LAYERS], K[2 * HB_MAX_LAYERS], NT[2 * HB_MAX_LAYERS],
        nch[2 * HB_MAX_LAYERS], nj = 0;
    for (int l = 0; l < Q.n_layers; ++l) {
      W[nj] = params + P.w[l]; ldn[nj] = Q.k[l]; ldk[nj] = 1; sc[nj] = (l == 0 && d->feature_norm) ? params + P.fn_w : nullptr;
      N[nj] = Q.n[l]; K[nj] = Q.k[l]; NT[nj] = Q.tk_nt[l]; nch[nj] = Q.tk_chunks[l]; dst[nj] = prepared + Q.tk[l]; ++nj;
      if (l >= 1) {  // W^T images: rows = input feature k, reduction = output feature n
        W[nj] = params + P.w[l]; ldn[nj] = 1; ldk[nj] = Q.k[l]; sc[nj] = nullptr; N[nj] = Q.k[l]; K[nj] = Q.n[l];
        NT[nj] = Q.tkt_nt[l]; nch[nj] = Q.tkt_chunks[l]; dst[nj] = prepared + Q.tkt[l]; ++nj;
      }
    }
    rc = launch_pack_umma_jobs(nj, W, ldn, ldk, sc, N, K, NT, nch, dst, st);
    if (rc) return rc;
  }
  if (Q.fz_ok) return launch_fused_pack(d, P, Q, params, prepared, st);
  return HB_OK;
}

}  // namespace hb

extern "C" {

int hb_version(void) { return HB_VERSION; }
const char* hb_last_error(void) { return hb::g_err; }
int hb_sync_check(void) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return hb::cuda_fail(e, "hb_sync_check");
  return HB_OK;
}

int hb_set_gemm_impl(int impl) {
  HB_CHECK_ARG(impl == 0 || impl == 1, "impl must be 0 (fp32 simt) or 1 (tcgen05 3xtf32)");
  hb::g_gemm_impl.store(impl);
  return HB_OK;
}
int hb_get_gemm_impl(void) { return hb::gemm_impl(); }

int hb_net_layout_of(const hb_net_desc* d, hb_net_layout* out) {
  HB_CHECK_ARG(out != nullptr, "out is NULL");
  return hb::make_layouts(d, nullptr, nullptr, out);
}

int hb_net_prepare(const hb_net_desc* d, const float* params, float* prepared, void* stream) {
  HB_CHECK_ARG(params && prepared, "NULL buffer");
  return hb::prepare_launch(d, params, prepared, (cudaStream_t)stream);
}
}
