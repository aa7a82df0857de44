// C-ABI entry points that sequence the kernels for one network over row chunks.
//
// Rows are processed in chunks of up to 2^20 (the workspace is sized for one chunk: ~3 KB per row at hidden 128,
// i.e. ~3 GB -- nothing against 180 GB of HBM3e).  Measured on B200 (profiles/chunk_sweep_r01.txt): L2-sized
// chunks of 32768 rows leave the GPU with 256 CTAs per launch -- 1.7 per SM, latency-bound at every kernel --
// and cost 94 ms per C2 update phase; whole-batch launches (819200 rows, 6400 CTAs) take 55 ms although the
// activations then stream through HBM.
#include <stdlib.h>

#include <atomic>

#include "common.cuh"
#include "kernels.cuh"
#include "rnn.cuh"
#include "trpo.cuh"

#include "fused_args.cuh"

namespace hb {

constexpr int64_t CHUNK_ROWS = (int64_t)1 << 20;   // rows per kernel launch

struct Work {
  float* x0;
  float* Z[HB_MAX_LAYERS];
  float* Y[HB_MAX_LAYERS];
  float* stats[HB_MAX_LAYERS];
  float* dA;
  float* dB;
  float* dwpart;   // [tc_dw_splits()][param total] split buffer of the tensor-core dW kernel (gradient mode)
  int ptotal;
  RnnWork rnn;     // GRU buffers (recurrent networks only)
};

// rows per launch: recurrent batches are never split (a chunk would have to cut every sequence)
static int64_t chunk_of(const hb_net_desc* d, int64_t rows) {
  if (rows < 1) return 1;
  return (d->rnn_layers || rows < CHUNK_ROWS) ? rows : CHUNK_ROWS;
}

// the sequence structure of a recurrent batch (RNNLayer.forward, rnn.py:22-81)
struct SeqCtx {
  const float* h0;      // [buffer rows, rnn_layers * h]; sequence j starts from row (index ? index[j] : j)
  const float* masks;   // [buffer rows]
  int64_t S;            // steps; batch rows are step-major, B = rows / S
  float* h_out;         // nullable [B, rnn_layers * h]
};

static int hmax_of(const PrepLayout& Q) {
  int m = 0;
  for (int l = 0; l < Q.n_layers; ++l) m = Q.n[l] > m ? Q.n[l] : m;
  return m;
}

static size_t base_floats(const PrepLayout& Q, int64_t ch, int mode, int ptotal) {
  size_t f = (size_t)ch * Q.kpad[0];
  const size_t hm = hmax_of(Q);
  if (mode == 0) return f + 2 * (size_t)ch * hm;
  for (int l = 0; l < Q.n_layers; ++l) f += 2 * (size_t)ch * Q.n[l] + (size_t)round_up((int)(2 * ch), 4);
  return f + 2 * (size_t)ch * hm + (size_t)round_up(tc_dw_splits() * ptotal, 4);
}

static size_t work_floats(const PrepLayout& Q, int64_t ch, int mode, int ptotal) {
  return base_floats(Q, ch, mode, ptotal) + rnn_work_floats(Q, ch, mode);
}

static int carve(const PrepLayout& Q, int64_t ch, int mode, void* ws, size_t ws_bytes, Work* w, int ptotal = 0) {
  if (work_floats(Q, ch, mode, ptotal) * sizeof(float) > ws_bytes || ws == nullptr) {
    set_error("workspace too small: need %zu bytes, have %zu", work_floats(Q, ch, mode, ptotal) * sizeof(float), ws_bytes);
    return HB_ERR_WORKSPACE;
  }
  w->ptotal = ptotal;
  w->dwpart = nullptr;
  float* p = (float*)ws;
  const size_t hm = hmax_of(Q);
  w->x0 = p; p += (size_t)ch * Q.kpad[0];
  if (mode == 0) {
    w->dA = p; p += (size_t)ch * hm;
    w->dB = p;
    for (int l = 0; l < Q.n_layers; ++l) { w->Z[l] = nullptr; w->stats[l] = nullptr; w->Y[l] = (l & 1) ? w->dB : w->dA; }
    return carve_rnn(Q, ch, 0, (float*)ws + base_floats(Q, ch, 0, ptotal), &w->rnn);
  }
  for (int l = 0; l < Q.n_layers; ++l) {
    w->Z[l] = p; p += (size_t)ch * Q.n[l];
    w->Y[l] = p; p += (size_t)ch * Q.n[l];
    w->stats[l] = p; p += (size_t)round_up((int)(2 * ch), 4);
  }
  w->dA = p; p += (size_t)ch * hm;
  w->dB = p; p += (size_t)ch * hm;
  w->dwpart = p;
  return carve_rnn(Q, ch, 1, (float*)ws + base_floats(Q, ch, 1, ptotal), &w->rnn);
}

static int trunk_forward(const hb_net_desc* d, const PrepLayout& Q, const float* prep, const float* obs,
                         const int32_t* index, int64_t c0, int64_t rows, const Work& w, cudaStream_t st);

// trunk (+ GRU + its LayerNorm): *feat = the head's input rows
static int features_forward(const hb_net_desc* d, const PrepLayout& Q, const float* prep, const float* obs,
                            const int32_t* index, int64_t c0, int64_t rows, const SeqCtx* seq, const Work& w,
                            cudaStream_t st, const float** feat) {
  int rc = trunk_forward(d, Q, prep, obs, index, c0, rows, w, st);
  if (rc) return rc;
  *feat = w.Y[Q.n_layers - 1];
  if (!d->rnn_layers) return HB_OK;
  if (seq == nullptr || seq->h0 == nullptr || seq->masks == nullptr || seq->S < 1 || rows % seq->S != 0) {
    set_error("recurrent network: the batch needs rnn_states, masks and a seq_len dividing its %lld rows", (long long)rows);
    return HB_ERR_INVALID;
  }
  rc = rnn_forward(Q, prep, *feat, seq->S, rows / seq->S, seq->h0, seq->masks, index, seq->h_out, w.rnn, st);
  *feat = w.rnn.out;
  return rc;
}

// recurrent networks: head wrote d/d(hs_top) into w.rnn.dtop -> BPTT -> LN/act backward of the last trunk block -> w.dA
static int rnn_to_trunk_backward(const hb_net_desc* d, const ParamLayout& P, const PrepLayout& Q, const float* params,
                                 const float* prep, float* grad, int64_t rows, const SeqCtx* seq, const Work& w,
                                 cudaStream_t st) {
  const int Lh = Q.n_layers;
  float* dX = nullptr;
  int rc = rnn_backward(P, Q, params, w.Y[Lh - 1], seq->S, rows / seq->S, grad, w.rnn, &dX, st);
  if (rc) return rc;
  return launch_ln_act_bwd(dX, w.Z[Lh - 1], w.stats[Lh - 1], prep + Q.lnw[Lh - 1], w.dA, grad + P.lnw[Lh - 1],
                           grad + P.lnb[Lh - 1], rows, Q.n[Lh - 1], d->activation, st);
}

// feature norm + trunk for `rows` rows starting at buffer row c0 (or index + c0)
static int trunk_forward(const hb_net_desc* d, const PrepLayout& Q, const float* prep, const float* obs,
                         const int32_t* index, int64_t c0, int64_t rows, const Work& w, cudaStream_t st) {
  const float* o = index ? obs : obs + c0 * d->in_dim;
  const int32_t* idx = index ? index + c0 : nullptr;
  int rc = launch_feat_norm(o, d->in_dim, idx, rows, d->feature_norm, w.x0, Q.kpad[0], st);
  if (rc) return rc;
  const float* x = w.x0;
  int ldx = Q.kpad[0];
  for (int l = 0; l < Q.n_layers; ++l) {
    if (gemm_impl() != 0)
      rc = launch_tc_linear_ln_fwd(d->activation, x, ldx, prep + Q.tk[l], Q.tk_chunks[l],
                                   prep + Q.bias[l], prep + Q.lnw[l], prep + Q.lnb[l], w.Z[l], w.Y[l], w.stats[l], rows,
                                   Q.n[l], Q.kpad[l], st);
    else
      rc = launch_linear_ln_fwd(d->activation, x, ldx, prep + Q.wt[l], prep + Q.bias[l], prep + Q.lnw[l], prep + Q.lnb[l],
                                w.Z[l], w.Y[l], w.stats[l], rows, Q.n[l], Q.kpad[l], st);
    if (rc) return rc;
    x = w.Y[l];
    ldx = Q.n[l];
  }
  return HB_OK;
}

// backward through the trunk given d(loss)/d(features) in w.dA
static int trunk_backward(const hb_net_desc* d, const ParamLayout& P, const PrepLayout& Q, const float* params,
                          const float* prep, float* grad, int64_t rows, const Work& w, cudaStream_t st) {
  const int L = Q.n_layers;
  float* dcur = w.dA;
  float* dnext = w.dB;
  int rc = HB_OK;  // the LN + activation backward of the last block is fused into the head kernel (w.dA already holds dZ_L)
  const int impl = gemm_impl();
  for (int l = L - 1; l >= 1; --l) {
    if (impl != 0)
      rc = launch_tc_dw_accum(dcur, Q.n[l], w.Y[l - 1], Q.n[l - 1], Q.k[l], w.dwpart + P.w[l], grad + P.b[l], rows,
                              w.ptotal, st);
    else
      rc = launch_dw_accum(dcur, Q.n[l], w.Y[l - 1], Q.n[l - 1], Q.k[l], grad + P.w[l], grad + P.b[l], rows, st);
    if (rc) return rc;
    if (impl != 0)
      rc = launch_tc_dx_ln_bwd(d->activation, dcur, Q.n[l], prep + Q.tkt[l], Q.tkt_chunks[l], w.Z[l - 1],
                               w.stats[l - 1], prep + Q.lnw[l - 1], dnext, grad + P.lnw[l - 1], grad + P.lnb[l - 1], rows,
                               Q.n[l - 1], w.dwpart - grad, w.ptotal, st);
    else
      rc = launch_dx_ln_bwd(d->activation, dcur, Q.n[l], params + P.w[l], w.Z[l - 1], w.stats[l - 1], prep + Q.lnw[l - 1],
                            dnext, grad + P.lnw[l - 1], grad + P.lnb[l - 1], rows, Q.n[l - 1], st);
    if (rc) return rc;
    float* t = dcur; dcur = dnext; dnext = t;
  }
  if (impl != 0)
    return launch_tc_dw_accum(dcur, Q.n[0], w.x0, Q.kpad[0], Q.k[0], w.dwpart + P.w[0], grad + P.b[0], rows, w.ptotal, st);
  return launch_dw_accum(dcur, Q.n[0], w.x0, Q.kpad[0], Q.k[0], grad + P.w[0], grad + P.b[0], rows, st);
}

static int check_net(const hb_net_desc* d, ParamLayout* P, PrepLayout* Q, hb_net_layout* L, int want_policy) {
  int rc = make_layouts(d, P, Q, L);
  if (rc) return rc;
  if (want_policy == 1 && d->head == HB_HEAD_VALUE) { set_error("expected a policy head"); return HB_ERR_INVALID; }
  if (want_policy == 0 && d->head != HB_HEAD_VALUE) { set_error("expected a value head"); return HB_ERR_INVALID; }
  return HB_OK;
}

static void head_base(const hb_net_desc* d, const PrepLayout& Q, const float* prep, HeadArgs* a) {
  memset(a, 0, sizeof(*a));
  a->h = Q.n[Q.n_layers - 1];
  a->out = d->out_dim;
  a->hw = prep + Q.hw;
  a->hbias = prep + Q.hbias;
  a->log_std = prep + Q.log_std;
  a->std_x = d->std_x_coef;
  a->std_y = d->std_y_coef;
}

// advance the buffer-row-indexed pointers of a batch to chunk start c0 (identity index only)
static void head_batch(const hb_net_desc* d, const hb_actor_batch* b, int64_t c0, int64_t rows, HeadArgs* a) {
  const int ad = d->head == HB_HEAD_DISCRETE ? 1 : d->out_dim;
  const int64_t o = b->index ? 0 : c0;
  a->rows = rows;
  a->index = b->index ? b->index + c0 : nullptr;
  a->actions = b->actions ? b->actions + o * ad : nullptr;
  a->avail = b->avail ? b->avail + o * d->out_dim : nullptr;
  a->old_logp = b->old_logp ? b->old_logp + o * ad : nullptr;
  a->adv = b->adv ? b->adv + o : nullptr;
  a->factor = b->factor ? b->factor + o : nullptr;
  a->active = b->active ? b->active + o : nullptr;
}

}  // namespace hb

extern "C" {

size_t hb_workspace_bytes(const hb_net_desc* d, int64_t rows, int mode) {
  hb::PrepLayout Q;
  hb::ParamLayout P;
  if (hb::make_layouts(d, &P, &Q, nullptr)) return 0;
  const int64_t ch = hb::chunk_of(d, rows);
  return hb::work_floats(Q, ch, mode, P.total) * sizeof(float);
}

static int policy_act_impl(const hb_net_desc* d, const float* prepared, const float* obs, int64_t rows,
                           const float* avail, const float* h_in, const float* masks, int deterministic, uint64_t seed,
                           uint64_t offset, const uint64_t* offset_base, float* actions, float* logp, float* h_out,
                           void* ws, size_t ws_bytes, void* stream) {
  using namespace hb;
  HB_CHECK_ARG(prepared && obs && actions && logp && rows >= 0, "bad argument");
  PrepLayout Q;
  int rc = check_net(d, nullptr, &Q, nullptr, 1);
  if (rc) return rc;
  HB_CHECK_ARG(!d->rnn_layers || (h_in && masks && h_out), "recurrent policy: rnn_states, masks and rnn_states_out are required");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t ch = chunk_of(d, rows);
  if (rows == 0) return HB_OK;
  if (!d->rnn_layers && fused_enabled()) {   // the same tensor-core kernel as hb_rollout_collect (one net)
    fz::ActArgs F;
    memset(&F, 0, sizeof(F));
    bool ok = false;
    if ((rc = fused_act_fill(&F.net[0], d, prepared, obs, avail, actions, logp, seed, rows, &ok))) return rc;
    if (ok) {
      F.n_nets = 1; F.H = d->hidden[0]; F.act = d->activation; F.deterministic = deterministic;
      F.offset = offset; F.offset_base = reinterpret_cast<const unsigned long long*>(offset_base);
      return launch_fused_act(F, st);
    }
  }
  Work w;
  if ((rc = carve(Q, ch, 0, ws, ws_bytes, &w))) return rc;
  const int ad = d->head == HB_HEAD_DISCRETE ? 1 : d->out_dim;
  for (int64_t c0 = 0; c0 < rows; c0 += ch) {
    const int64_t n = rows - c0 < ch ? rows - c0 : ch;
    SeqCtx seq = {h_in, masks, 1, h_out};  // one step: S = 1, every row its own sequence (rnn.py:24-32)
    const float* feat = nullptr;
    if ((rc = features_forward(d, Q, prepared, obs, nullptr, c0, n, d->rnn_layers ? &seq : nullptr, w, st, &feat))) return rc;
    HeadArgs a;
    head_base(d, Q, prepared, &a);
    a.feat = feat;
    a.rows = n;
    a.avail = avail ? avail + c0 * d->out_dim : nullptr;
    a.deterministic = deterministic;
    a.seed = seed;
    a.offset = offset + (uint64_t)c0 * 0x9E3779B97F4A7C15ull;  // distinct Philox streams per chunk
    a.offset_base = reinterpret_cast<const unsigned long long*>(offset_base);
    a.actions_out = actions + c0 * ad;
    a.logp_out = logp + c0 * ad;
    if ((rc = launch_policy_head(d->head, MODE_ACT, a, st))) return rc;
  }
  return HB_OK;
}

static int value_forward_impl(const hb_net_desc* d, const float* prepared, const float* cent_obs, int64_t rows,
                              const float* h_in, const float* masks, float* values, float* h_out, void* ws,
                              size_t ws_bytes, void* stream) {
  using namespace hb;
  HB_CHECK_ARG(prepared && cent_obs && values && rows >= 0, "bad argument");
  PrepLayout Q;
  int rc = check_net(d, nullptr, &Q, nullptr, 0);
  if (rc) return rc;
  HB_CHECK_ARG(!d->rnn_layers || (h_in && masks && h_out), "recurrent critic: rnn_states, masks and rnn_states_out are required");
  cudaStream_t st = (cudaStream_t)stream;
  if (rows == 0) return HB_OK;
  if (!d->rnn_layers && fused_enabled()) {
    fz::ActArgs F;
    memset(&F, 0, sizeof(F));
    bool ok = false;
    if ((rc = fused_act_fill(&F.net[0], d, prepared, cent_obs, nullptr, values, nullptr, 0ull, rows, &ok))) return rc;
    if (ok) {
      F.n_nets = 1; F.H = d->hidden[0]; F.act = d->activation;
      return launch_fused_act(F, st);
    }
  }
  const int64_t ch = chunk_of(d, rows);
  Work w;
  if ((rc = carve(Q, ch, 0, ws, ws_bytes, &w))) return rc;
  for (int64_t c0 = 0; c0 < rows; c0 += ch) {
    const int64_t n = rows - c0 < ch ? rows - c0 : ch;
    SeqCtx seq = {h_in, masks, 1, h_out};
    const float* feat = nullptr;
    if ((rc = features_forward(d, Q, prepared, cent_obs, nullptr, c0, n, d->rnn_layers ? &seq : nullptr, w, st, &feat))) return rc;
    ValueArgs a;
    memset(&a, 0, sizeof(a));
    a.feat = feat;
    a.h = Q.n[Q.n_layers - 1];
    a.hw = prepared + Q.hw;
    a.hbias = prepared + Q.hbias;
    a.rows = n;
    a.values_out = values + c0;
    if ((rc = launch_value_head(0, a, st))) return rc;
  }
  return HB_OK;
}

int hb_policy_act(const hb_net_desc* d, const float* prepared, const float* obs, int64_t rows, const float* avail,
                  int deterministic, uint64_t seed, uint64_t offset, float* actions, float* logp, void* ws,
                  size_t ws_bytes, void* stream) {
  return policy_act_impl(d, prepared, obs, rows, avail, nullptr, nullptr, deterministic, seed, offset, nullptr, actions,
                         logp, nullptr, ws, ws_bytes, stream);
}

int hb_policy_act_rnn(const hb_net_desc* d, const float* prepared, const float* obs, int64_t rows, const float* avail,
                      const float* rnn_states, const float* masks, int deterministic, uint64_t seed, uint64_t offset,
                      const uint64_t* offset_base, float* actions, float* logp, float* rnn_states_out, void* ws,
                      size_t ws_bytes, void* stream) {
  return policy_act_impl(d, prepared, obs, rows, avail, rnn_states, masks, deterministic, seed, offset, offset_base, actions,
                         logp, rnn_states_out, ws, ws_bytes, stream);
}

int hb_value_forward(const hb_net_desc* d, const float* prepared, const float* cent_obs, int64_t rows, float* values,
                     void* ws, size_t ws_bytes, void* stream) {
  return value_forward_impl(d, prepared, cent_obs, rows, nullptr, nullptr, values, nullptr, ws, ws_bytes, stream);
}

int hb_value_forward_rnn(const hb_net_desc* d, const float* prepared, const float* cent_obs, int64_t rows,
                         const float* rnn_states, const float* masks, float* values, float* rnn_states_out, void* ws,
                         size_t ws_bytes, void* stream) {
  return value_forward_impl(d, prepared, cent_obs, rows, rnn_states, masks, values, rnn_states_out, ws, ws_bytes, stream);
}

int hb_policy_evaluate(const hb_net_desc* d, const float* prepared, const hb_actor_batch* b, float* logp_out,
                       const float* logp_ref, float* factor_inout, int action_aggregation_prod, void* ws,
                       size_t ws_bytes, void* stream) {
  using namespace hb;
  HB_CHECK_ARG(prepared && b && b->obs && b->actions && b->rows >= 0, "bad argument");
  HB_CHECK_ARG(!factor_inout || (logp_ref && !b->index), "factor update needs logp_ref and an identity batch");
  PrepLayout Q;
  int rc = check_net(d, nullptr, &Q, nullptr, 1);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t rows = b->rows;
  if (rows == 0) return HB_OK;
  if (Q.fz_ok && fused_enabled()) {  // one fused launch: feature norm -> trunk -> head, nothing round-trips HBM
    ParamLayout P;
    if ((rc = make_layouts(d, &P, nullptr, nullptr))) return rc;
    fz::Args fa;
    memset(&fa, 0, sizeof(fa));
    fa.obs = b->obs; fa.index = b->index; fa.rows = rows;
    fa.actions = b->actions; fa.avail = b->avail;
    fa.logp_out = logp_out; fa.logp_ref = logp_ref; fa.factor_inout = factor_inout;
    fa.agg_prod = action_aggregation_prod;
    return launch_fused_update(d, Q, P, prepared, fa, 1, nullptr, st);
  }
  const int64_t ch = chunk_of(d, rows);
  Work w;
  if ((rc = carve(Q, ch, 0, ws, ws_bytes, &w))) return rc;
  const int ad = d->head == HB_HEAD_DISCRETE ? 1 : d->out_dim;
  for (int64_t c0 = 0; c0 < rows; c0 += ch) {
    const int64_t n = rows - c0 < ch ? rows - c0 : ch;
    SeqCtx seq = {b->rnn_states, b->masks, b->seq_len, nullptr};
    const float* feat = nullptr;
    if ((rc = features_forward(d, Q, prepared, b->obs, b->index, c0, n, d->rnn_layers ? &seq : nullptr, w, st, &feat))) return rc;
    HeadArgs a;
    head_base(d, Q, prepared, &a);
    head_batch(d, b, c0, n, &a);
    a.feat = feat;
    a.logp_out = logp_out ? logp_out + c0 * ad : nullptr;
    a.logp_ref = logp_ref ? logp_ref + c0 * ad : nullptr;
    a.factor_inout = factor_inout ? factor_inout + c0 : nullptr;
    a.agg_prod = action_aggregation_prod;
    if ((rc = launch_policy_head(d->head, MODE_EVAL, a, st))) return rc;
  }
  return HB_OK;
}

int hb_ppo_actor_grad(const hb_net_desc* d, const float* params, const float* prepared, const hb_actor_batch* b,
                      const hb_ppo_hyper* h, const double* norm3, float* grad, double* scalars, void* ws,
                      size_t ws_bytes, void* stream) {
  return hb_ppo_actor_grad_logp(d, params, prepared, b, h, norm3, grad, scalars, nullptr, ws, ws_bytes, stream);
}

int hb_ppo_actor_grad_logp(const hb_net_desc* d, const float* params, const float* prepared, const hb_actor_batch* b,
                           const hb_ppo_hyper* h, const double* norm3, float* grad, double* scalars, float* logp_out, void* ws,
                           size_t ws_bytes, void* stream) {
  using namespace hb;
  HB_CHECK_ARG(params && prepared && b && h && norm3 && grad && scalars, "NULL argument");
  HB_CHECK_ARG(b->obs && b->actions && b->old_logp && b->adv && b->active && b->rows >= 0, "incomplete batch");
  HB_CHECK_ARG(!logp_out || !b->index, "logp_out needs an identity batch (rows of the batch = rows of logp_out)");
  ParamLayout P;
  PrepLayout Q;
  hb_net_layout L;
  int rc = check_net(d, &P, &Q, &L, 1);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (Q.fz_ok && fused_enabled() && b->rows > 0) {
    // fused forward + loss + backward: the workspace only holds the per-CTA slots of the weight-gradient sums
    const size_t need = (size_t)fused_max_slots() * L.total * sizeof(float);
    if (ws == nullptr || ws_bytes < need) { set_error("hb_ppo_actor_grad: workspace too small: need %zu bytes, have %zu", need, ws_bytes); return HB_ERR_WORKSPACE; }
    fz::Args fa;
    memset(&fa, 0, sizeof(fa));
    fa.obs = b->obs; fa.index = b->index; fa.rows = b->rows;
    fa.actions = b->actions; fa.avail = b->avail; fa.old_logp = b->old_logp; fa.adv = b->adv; fa.factor = b->factor; fa.active = b->active;
    fa.clip = h->clip_param; fa.entropy_coef = h->entropy_coef; fa.use_active = h->use_policy_active_masks;
    fa.use_clip = h->use_clip; fa.agg_prod = h->action_aggregation_prod;
    fa.part = (float*)ws; fa.part_stride = L.total; fa.scalars = scalars;
    fa.logp_out = logp_out;
    int slots = 0;
    if ((rc = launch_fused_update(d, Q, P, prepared, fa, 0, &slots, st))) return rc;
    return launch_fused_finish(d, P, params, grad, (const float*)ws, slots, L.total, norm3, 1.0, st);
  }
  if (logp_out && b->rows > 0) {  // layer-wise kernels: a separate forward sweep writes the log-probs
    rc = hb_policy_evaluate(d, prepared, b, logp_out, nullptr, nullptr, h->action_aggregation_prod, ws, ws_bytes, stream);
    if (rc) return rc;
  }
  cudaError_t ce = cudaMemsetAsync(grad, 0, (size_t)L.total * sizeof(float), st);
  if (ce != cudaSuccess) return cuda_fail(ce, "hb_ppo_actor_grad(memset)");
  const int64_t rows = b->rows;
  if (rows == 0) return HB_OK;
  const int64_t ch = chunk_of(d, rows);
  Work w;
  if ((rc = carve(Q, ch, 1, ws, ws_bytes, &w, L.total))) return rc;
  {
    ce = cudaMemsetAsync(w.dwpart, 0, (size_t)tc_dw_splits() * L.total * sizeof(float), st);
    if (ce != cudaSuccess) return cuda_fail(ce, "hb_ppo_actor_grad(memset split buffer)");
  }
  const bool rnn = d->rnn_layers != 0;
  for (int64_t c0 = 0; c0 < rows; c0 += ch) {
    const int64_t n = rows - c0 < ch ? rows - c0 : ch;
    SeqCtx seq = {b->rnn_states, b->masks, b->seq_len, nullptr};
    const float* feat = nullptr;
    if ((rc = features_forward(d, Q, prepared, b->obs, b->index, c0, n, rnn ? &seq : nullptr, w, st, &feat))) return rc;
    HeadArgs a;
    head_base(d, Q, prepared, &a);
    head_batch(d, b, c0, n, &a);
    a.feat = feat;
    a.agg_prod = h->action_aggregation_prod;
    a.clip = h->clip_param;
    a.entropy_coef = h->entropy_coef;
    a.use_active = h->use_policy_active_masks;
    a.use_clip = h->use_clip;
    a.norm3 = norm3;
    a.dfeat = w.dA;
    a.g_hw = grad + P.hw;
    a.g_hbias = grad + P.hbias;
    a.g_log_std = d->head == HB_HEAD_BOX ? grad + P.log_std : nullptr;
    a.scalars = scalars;
    a.ln_z = w.Z[Q.n_layers - 1]; a.ln_stats = w.stats[Q.n_layers - 1]; a.ln_w = prepared + Q.lnw[Q.n_layers - 1];
    a.g_ln_w = grad + P.lnw[Q.n_layers - 1]; a.g_ln_b = grad + P.lnb[Q.n_layers - 1]; a.ln_act = d->activation;
    if (rnn) {  // the head's input is LayerNorm(GRU output): fuse that LN's backward (identity activation) instead
      a.dfeat = w.rnn.dtop;
      a.ln_z = w.rnn.hs[d->rnn_layers - 1]; a.ln_stats = w.rnn.stats; a.ln_w = prepared + Q.rnn_lnw;
      a.g_ln_w = grad + P.rnn_lnw; a.g_ln_b = grad + P.rnn_lnb; a.ln_act = HB_ACT_IDENTITY;
    }
    a.part_delta = w.dwpart - grad; a.part_stride = w.ptotal;
    if ((rc = launch_policy_head(d->head, MODE_GRAD, a, st))) return rc;
    if (rnn && (rc = rnn_to_trunk_backward(d, P, Q, params, prepared, grad, n, &seq, w, st))) return rc;
    if ((rc = trunk_backward(d, P, Q, params, prepared, grad, n, w, st))) return rc;
  }
  if ((rc = launch_dw_reduce(grad, w.dwpart, L.total, st))) return rc;
  return launch_featnorm_fold(d, params, grad, st);
}

int hb_value_grad(const hb_net_desc* d, const float* params, const float* prepared, const hb_critic_batch* b,
                  const hb_value_hyper* h, const float* vn_state, double inv_count, float* grad, double* scalars,
                  void* ws, size_t ws_bytes, void* stream) {
  using namespace hb;
  HB_CHECK_ARG(params && prepared && b && h && grad && scalars, "NULL argument");
  HB_CHECK_ARG(b->share_obs && b->value_preds && b->returns && b->rows >= 0, "incomplete batch");
  ParamLayout P;
  PrepLayout Q;
  hb_net_layout L;
  int rc = check_net(d, &P, &Q, &L, 0);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (Q.fz_ok && fused_enabled() && b->rows > 0) {
    const size_t need = (size_t)fused_max_slots() * L.total * sizeof(float);
    if (ws == nullptr || ws_bytes < need) { set_error("hb_value_grad: workspace too small: need %zu bytes, have %zu", need, ws_bytes); return HB_ERR_WORKSPACE; }
    fz::Args fa;
    memset(&fa, 0, sizeof(fa));
    fa.obs = b->share_obs; fa.index = b->index; fa.rows = b->rows;
    fa.value_preds = b->value_preds; fa.returns = b->returns; fa.vn_state = vn_state;
    fa.clip = h->clip_param; fa.huber_delta = h->huber_delta; fa.vcoef = h->value_loss_coef;
    fa.use_huber = h->use_huber_loss; fa.use_clipped = h->use_clipped_value_loss;
    fa.part = (float*)ws; fa.part_stride = L.total; fa.scalars = scalars;
    int slots = 0;
    if ((rc = launch_fused_update(d, Q, P, prepared, fa, 0, &slots, st))) return rc;
    return launch_fused_finish(d, P, params, grad, (const float*)ws, slots, L.total, nullptr, inv_count, st);
  }
  cudaError_t ce = cudaMemsetAsync(grad, 0, (size_t)L.total * sizeof(float), st);
  if (ce != cudaSuccess) return cuda_fail(ce, "hb_value_grad(memset)");
  const int64_t rows = b->rows;
  if (rows == 0) return HB_OK;
  const int64_t ch = chunk_of(d, rows);
  Work w;
  if ((rc = carve(Q, ch, 1, ws, ws_bytes, &w, L.total))) return rc;
  {
    ce = cudaMemsetAsync(w.dwpart, 0, (size_t)tc_dw_splits() * L.total * sizeof(float), st);
    if (ce != cudaSuccess) return cuda_fail(ce, "hb_value_grad(memset split buffer)");
  }
  const bool rnn = d->rnn_layers != 0;
  for (int64_t c0 = 0; c0 < rows; c0 += ch) {
    const int64_t n = rows - c0 < ch ? rows - c0 : ch;
    SeqCtx seq = {b->rnn_states, b->masks, b->seq_len, nullptr};
    const float* feat = nullptr;
    if ((rc = features_forward(d, Q, prepared, b->share_obs, b->index, c0, n, rnn ? &seq : nullptr, w, st, &feat))) return rc;
    ValueArgs a;
    memset(&a, 0, sizeof(a));
    a.feat = feat;
    a.h = Q.n[Q.n_layers - 1];
    a.hw = prepared + Q.hw;
    a.hbias = prepared + Q.hbias;
    a.rows = n;
    const int64_t o = b->index ? 0 : c0;
    a.index = b->index ? b->index + c0 : nullptr;
    a.value_preds = b->value_preds + o;
    a.returns = b->returns + o;
    a.vn_state = vn_state;
    a.clip = h->clip_param;
    a.huber_delta = h->huber_delta;
    a.coef = (float)((double)h->value_loss_coef * inv_count);
    a.use_huber = h->use_huber_loss;
    a.use_clipped = h->use_clipped_value_loss;
    a.dfeat = w.dA;
    a.g_hw = grad + P.hw;
    a.g_hbias = grad + P.hbias;
    a.scalars = scalars;
    a.ln_z = w.Z[Q.n_layers - 1]; a.ln_stats = w.stats[Q.n_layers - 1]; a.ln_w = prepared + Q.lnw[Q.n_layers - 1];
    a.g_ln_w = grad + P.lnw[Q.n_layers - 1]; a.g_ln_b = grad + P.lnb[Q.n_layers - 1]; a.ln_act = d->activation;
    if (rnn) {
      a.dfeat = w.rnn.dtop;
      a.ln_z = w.rnn.hs[d->rnn_layers - 1]; a.ln_stats = w.rnn.stats; a.ln_w = prepared + Q.rnn_lnw;
      a.g_ln_w = grad + P.rnn_lnw; a.g_ln_b = grad + P.rnn_lnb; a.ln_act = HB_ACT_IDENTITY;
    }
    a.part_delta = w.dwpart - grad; a.part_stride = w.ptotal;
    if ((rc = launch_value_head(1, a, st))) return rc;
    if (rnn && (rc = rnn_to_trunk_backward(d, P, Q, params, prepared, grad, n, &seq, w, st))) return rc;
    if ((rc = trunk_backward(d, P, Q, params, prepared, grad, n, w, st))) return rc;
  }
  if ((rc = launch_dw_reduce(grad, w.dwpart, L.total, st))) return rc;
  return launch_featnorm_fold(d, params, grad, st);
}

/* ------------------------------------------------------------------ trust-region (HATRPO) update */
namespace {
struct TrpoExtra { float* tprep; float* yd[2]; float* ttiles; };

// tangent-prepared weights, two tangent activation buffers, GRU tangent buffers, and (tensor-core tangent block) the
// UMMA images of the tangent weights -- same size as the forward images
size_t trpo_extra_floats(const hb::PrepLayout& Q, int64_t ch) {
  return (size_t)hb::round_up(Q.tk[0], 4) + 2 * (size_t)ch * hb::hmax_of(Q) + hb::rnn_jvp_floats(Q, ch) +
         (size_t)hb::round_up(Q.total - Q.tk[0], 4);
}

// 0 = FP32 FFMA tangent block, 1 = tcgen05 tangent block (both GPU-verified against each other:
// tests/test_gpu_zz_wide_heads.py::test_tensor_core_tangent_block_equals_ffma).  Env HB_TRPO_JVP_IMPL overrides the default.
int trpo_jvp_default() {
  const char* e = getenv("HB_TRPO_JVP_IMPL");
  return e ? (atoi(e) != 0) : 1;   // default since round 2: the tcgen05 tangent block (C2T 4.57 -> 5.73 M env-steps/s)
}
std::atomic<int> g_trpo_jvp_impl{trpo_jvp_default()};


}  // namespace

size_t hb_trpo_workspace_bytes(const hb_net_desc* d, int64_t rows) {
  hb::PrepLayout Q;
  hb::ParamLayout P;
  if (hb::make_layouts(d, &P, &Q, nullptr)) return 0;
  const int64_t ch = hb::chunk_of(d, rows);
  return (hb::work_floats(Q, ch, 1, P.total) + trpo_extra_floats(Q, ch)) * sizeof(float);
}

int hb_trpo_old_dist(const hb_net_desc* d, const float* prepared, const hb_actor_batch* b, float* old_dist, void* ws,
                     size_t ws_bytes, void* stream) {
  using namespace hb;
  HB_CHECK_ARG(prepared && b && b->obs && old_dist && b->rows >= 0, "bad argument");
  PrepLayout Q;
  int rc = check_net(d, nullptr, &Q, nullptr, 1);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t rows = b->rows;
  if (rows == 0) return HB_OK;
  const int64_t ch = chunk_of(d, rows);
  Work w;
  if ((rc = carve(Q, ch, 0, ws, ws_bytes, &w))) return rc;
  for (int64_t c0 = 0; c0 < rows; c0 += ch) {
    const int64_t n = rows - c0 < ch ? rows - c0 : ch;
    SeqCtx seq = {b->rnn_states, b->masks, b->seq_len, nullptr};
    const float* feat = nullptr;
    if ((rc = features_forward(d, Q, prepared, b->obs, b->index, c0, n, d->rnn_layers ? &seq : nullptr, w, st, &feat))) return rc;
    TrpoHeadArgs a;
    memset(&a, 0, sizeof(a));
    a.feat = feat;
    a.h = Q.n[Q.n_layers - 1]; a.out = d->out_dim;
    a.hw = prepared + Q.hw; a.hbias = prepared + Q.hbias; a.log_std = prepared + Q.log_std;
    a.std_x = d->std_x_coef; a.std_y = d->std_y_coef;
    a.rows = n;
    a.index = b->index ? b->index + c0 : nullptr;
    a.avail = b->avail ? b->avail + (b->index ? 0 : c0) * d->out_dim : nullptr;
    a.old_dist_out = old_dist + c0 * d->out_dim;
    if ((rc = launch_trpo_head(d->head, TR_OLD, a, st))) return rc;
  }
  return HB_OK;
}

int hb_trpo_fvp(const hb_net_desc* d, const float* params, const float* prepared, const hb_actor_batch* b,
                const float* old_dist, const float* v, double inv_rows, int reuse_forward, float* out, void* ws,
                size_t ws_bytes, void* stream) {
  using namespace hb;
  HB_CHECK_ARG(params && prepared && b && b->obs && old_dist && v && out && b->rows >= 0, "bad argument");
  ParamLayout P;
  PrepLayout Q;
  hb_net_layout L;
  int rc = check_net(d, &P, &Q, &L, 1);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t ce = cudaMemsetAsync(out, 0, (size_t)L.total * sizeof(float), st);
  if (ce != cudaSuccess) return cuda_fail(ce, "hb_trpo_fvp(memset)");
  const int64_t rows = b->rows;
  if (rows == 0) return HB_OK;
  const int64_t ch = chunk_of(d, rows);
  const bool rnn = d->rnn_layers != 0;
  const size_t base = work_floats(Q, ch, 1, L.total);
  if ((base + trpo_extra_floats(Q, ch)) * sizeof(float) > ws_bytes || ws == nullptr) {
    set_error("hb_trpo_fvp: workspace too small: need %zu bytes, have %zu", (base + trpo_extra_floats(Q, ch)) * sizeof(float), ws_bytes);
    return HB_ERR_WORKSPACE;
  }
  Work w;
  if ((rc = carve(Q, ch, 1, ws, base * sizeof(float), &w, L.total))) return rc;
  TrpoExtra x;
  x.tprep = (float*)ws + base;
  x.yd[0] = x.tprep + round_up(Q.tk[0], 4);
  x.yd[1] = x.yd[0] + (size_t)ch * hmax_of(Q);
  RnnJvpWork jw;
  carve_rnn_jvp(Q, ch, x.yd[1] + (size_t)ch * hmax_of(Q), &jw);
  x.ttiles = x.yd[1] + (size_t)ch * hmax_of(Q) + rnn_jvp_floats(Q, ch);
  const bool tc_jvp = g_trpo_jvp_impl.load(std::memory_order_relaxed) == 1 && gemm_impl() != 0;
  ce = cudaMemsetAsync(w.dwpart, 0, (size_t)tc_dw_splits() * L.total * sizeof(float), st);
  if (ce != cudaSuccess) return cuda_fail(ce, "hb_trpo_fvp(memset split buffer)");
  if ((rc = launch_tangent_prepare(d, P, Q, params, v, x.tprep, st))) return rc;
  const int Lh = Q.n_layers;
  if (tc_jvp) {  // UMMA images of the tangent weights (W^T layout of tprep: src(n, k) = wt[k * n_l + n])
    for (int l = 0; l < Lh; ++l)
      if ((rc = launch_pack_umma_tiles(x.tprep + Q.wt[l], 1, Q.n[l], nullptr, Q.n[l], Q.k[l], Q.tk_nt[l], Q.tk_chunks[l],
                                       x.ttiles + (Q.tk[l] - Q.tk[0]), st)))
        return rc;
  }
  for (int64_t c0 = 0; c0 < rows; c0 += ch) {
    const int64_t n = rows - c0 < ch ? rows - c0 : ch;
    SeqCtx seq = {b->rnn_states, b->masks, b->seq_len, nullptr};
    const float* feat = nullptr;
    if (reuse_forward && ch == rows) {
      // the 11 products of one update share parameters and batch: the activations (and the GRU's saved gates) of the
      // previous hb_trpo_fvp call are still in the workspace
      feat = rnn ? w.rnn.out : w.Y[Lh - 1];
    } else if ((rc = features_forward(d, Q, prepared, b->obs, b->index, c0, n, rnn ? &seq : nullptr, w, st, &feat))) {
      return rc;
    }
    // tangent pass through the trunk (the normalised observations carry no tangent: their affine is folded into layer 0)
    const float* xin = w.x0;
    const float* xd = nullptr;
    int ldx = Q.kpad[0];
    for (int l = 0; l < Lh; ++l) {
      float* yd = x.yd[l & 1];
      if (tc_jvp)
        rc = launch_tc_jvp_linear_ln(d->activation, xin, ldx, xd, prepared + Q.tk[l],
                                     x.ttiles + (Q.tk[l] - Q.tk[0]), Q.tk_chunks[l], x.tprep + Q.bias[l],
                                     prepared + Q.lnw[l], x.tprep + Q.lnw[l], x.tprep + Q.lnb[l], w.Z[l], w.stats[l], yd, n,
                                     Q.n[l], Q.kpad[l], st);
      else
        rc = launch_jvp_linear_ln(d->activation, xin, ldx, xd, prepared + Q.wt[l], x.tprep + Q.wt[l], x.tprep + Q.bias[l],
                                  prepared + Q.lnw[l], x.tprep + Q.lnw[l], x.tprep + Q.lnb[l], w.Z[l], w.stats[l], yd, n,
                                  Q.n[l], Q.kpad[l], st);
      if (rc) return rc;
      xin = w.Y[l]; xd = yd; ldx = Q.n[l];
    }
    if (rnn) {  // tangent through the GRU and its LayerNorm (the forward pass above saved the gates)
      if ((rc = rnn_jvp_forward(Q, prepared, x.tprep, w.Y[Lh - 1], xd, seq.S, n / seq.S, w.rnn, jw, st))) return rc;
      xd = jw.outd;
    }
    TrpoHeadArgs a;
    memset(&a, 0, sizeof(a));
    a.feat = feat; a.featd = xd;
    a.h = Q.n[Lh - 1]; a.out = d->out_dim;
    a.hw = prepared + Q.hw; a.hbias = prepared + Q.hbias; a.log_std = prepared + Q.log_std;
    a.hwd = x.tprep + Q.hw; a.hbd = x.tprep + Q.hbias;
    a.std_x = d->std_x_coef; a.std_y = d->std_y_coef;
    a.rows = n;
    a.index = b->index ? b->index + c0 : nullptr;
    a.avail = b->avail ? b->avail + (b->index ? 0 : c0) * d->out_dim : nullptr;
    a.old_dist = old_dist + c0 * d->out_dim;
    a.inv_rows = (float)inv_rows;
    a.dfeat = w.dA;
    a.g_hw = out + P.hw; a.g_hbias = out + P.hbias;
    a.ln_z = w.Z[Lh - 1]; a.ln_stats = w.stats[Lh - 1]; a.ln_w = prepared + Q.lnw[Lh - 1];
    a.g_ln_w = out + P.lnw[Lh - 1]; a.g_ln_b = out + P.lnb[Lh - 1]; a.ln_act = d->activation;
    if (rnn) {
      a.dfeat = w.rnn.dtop;
      a.ln_z = w.rnn.hs[d->rnn_layers - 1]; a.ln_stats = w.rnn.stats; a.ln_w = prepared + Q.rnn_lnw;
      a.g_ln_w = out + P.rnn_lnw; a.g_ln_b = out + P.rnn_lnb; a.ln_act = HB_ACT_IDENTITY;
    }
    a.part_delta = w.dwpart - out; a.part_stride = w.ptotal;
    if ((rc = launch_trpo_head(d->head, TR_FVP, a, st))) return rc;
    if (rnn && (rc = rnn_to_trunk_backward(d, P, Q, params, prepared, out, n, &seq, w, st))) return rc;
    if ((rc = trunk_backward(d, P, Q, params, prepared, out, n, w, st))) return rc;
  }
  if ((rc = launch_dw_reduce(out, w.dwpart, L.total, st))) return rc;
  return launch_featnorm_fold(d, params, out, st);
}

int hb_trpo_fvp_finish(const hb_net_desc* d, const float* params, const float* v, float* out, float damping,
                       void* stream) {
  using namespace hb;
  HB_CHECK_ARG(params && v && out, "NULL argument");
  ParamLayout P;
  hb_net_layout L;
  int rc = check_net(d, &P, nullptr, &L, 1);
  if (rc) return rc;
  const bool box = d->head == HB_HEAD_BOX;
  return launch_fvp_finish(out, v, params, damping, L.total, box ? P.log_std : 0, box ? d->out_dim : 0, d->std_x_coef,
                           (cudaStream_t)stream);
}

int hb_trpo_eval(const hb_net_desc* d, const float* prepared, const hb_actor_batch* b, const hb_ppo_hyper* h,
                 const float* old_dist, const float* params_old, double* scalars, void* ws, size_t ws_bytes,
                 void* stream) {
  using namespace hb;
  HB_CHECK_ARG(prepared && b && h && old_dist && params_old && scalars, "NULL argument");
  HB_CHECK_ARG(b->obs && b->actions && b->old_logp && b->adv && b->active && b->rows >= 0, "incomplete batch");
  ParamLayout P;
  PrepLayout Q;
  int rc = check_net(d, &P, &Q, nullptr, 1);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t rows = b->rows;
  if (rows == 0) return HB_OK;
  const int64_t ch = chunk_of(d, rows);
  Work w;
  if ((rc = carve(Q, ch, 0, ws, ws_bytes, &w))) return rc;
  const int ad = d->head == HB_HEAD_DISCRETE ? 1 : d->out_dim;
  for (int64_t c0 = 0; c0 < rows; c0 += ch) {
    const int64_t n = rows - c0 < ch ? rows - c0 : ch;
    SeqCtx seq = {b->rnn_states, b->masks, b->seq_len, nullptr};
    const float* feat = nullptr;
    if ((rc = features_forward(d, Q, prepared, b->obs, b->index, c0, n, d->rnn_layers ? &seq : nullptr, w, st, &feat))) return rc;
    const int64_t o = b->index ? 0 : c0;
    TrpoHeadArgs a;
    memset(&a, 0, sizeof(a));
    a.feat = feat;
    a.h = Q.n[Q.n_layers - 1]; a.out = d->out_dim;
    a.hw = prepared + Q.hw; a.hbias = prepared + Q.hbias; a.log_std = prepared + Q.log_std;
    a.std_x = d->std_x_coef; a.std_y = d->std_y_coef;
    a.rows = n;
    a.index = b->index ? b->index + c0 : nullptr;
    a.avail = b->avail ? b->avail + o * d->out_dim : nullptr;
    a.old_dist = old_dist + c0 * d->out_dim;
    a.actions = b->actions + o * ad;
    a.old_logp = b->old_logp + o * ad;
    a.adv = b->adv + o;
    a.factor = b->factor ? b->factor + o : nullptr;
    a.active = b->active + o;
    a.old_log_std = d->head == HB_HEAD_BOX ? params_old + P.log_std : nullptr;
    a.use_active = h->use_policy_active_masks;
    a.agg_prod = h->action_aggregation_prod;
    a.scalars = scalars;
    if ((rc = launch_trpo_head(d->head, TR_LS, a, st))) return rc;
  }
  return HB_OK;
}

int hb_trpo_cg_init(const float* b, float* x, float* r, float* p, float* state, int n, void* stream) {
  HB_CHECK_ARG(b && x && r && p && state && n > 0, "bad argument");
  return hb::launch_cg_init(b, x, r, p, state, n, (cudaStream_t)stream);
}

int hb_trpo_cg_step(float* p, const float* avp, float* x, float* r, float* state, int n, float residual_tol,
                    void* stream) {
  HB_CHECK_ARG(p && avp && x && r && state && n > 0, "bad argument");
  return hb::launch_cg_step(p, avp, x, r, state, n, residual_tol, (cudaStream_t)stream);
}

int hb_trpo_full_step(const float* x, const float* fx, const float* g, float kl_threshold, float* full_step,
                      double* out3, int n, void* stream) {
  HB_CHECK_ARG(x && fx && g && full_step && out3 && n > 0 && kl_threshold > 0.f, "bad argument");
  return hb::launch_full_step(x, fx, g, kl_threshold, full_step, out3, n, (cudaStream_t)stream);
}

int hb_trpo_apply_step(float* params, const float* params0, const float* full_step, float fraction, int n,
                       void* stream) {
  HB_CHECK_ARG(params && params0 && full_step && n > 0, "bad argument");
  return hb::launch_apply_step(params, params0, full_step, fraction, n, (cudaStream_t)stream);
}

int hb_set_trpo_jvp_impl(int impl) {
  HB_CHECK_ARG(impl == 0 || impl == 1, "impl must be 0 (FP32 FFMA tangent block) or 1 (tcgen05 tangent block)");
  g_trpo_jvp_impl.store(impl);
  return HB_OK;
}
int hb_get_trpo_jvp_impl(void) { return g_trpo_jvp_impl.load(); }

int hb_set_fused_update(int on) {
  hb::set_fused_enabled(on);
  return HB_OK;
}
int hb_get_fused_update(void) { return hb::fused_enabled() ? 1 : 0; }
int hb_fused_timing_enable(int on) { return hb::fused_timing_enable(on); }
int hb_fused_timing_read(unsigned long long* out) {
  HB_CHECK_ARG(out != nullptr, "NULL");
  return hb::fused_timing_read(out);
}

int hb_set_rnn_impl(int impl) {
  HB_CHECK_ARG(impl == 0 || impl == 1, "impl must be 0 (launch per step) or 1 (persistent recurrence)");
  hb::set_rnn_impl(impl);
  return HB_OK;
}
int hb_get_rnn_impl(void) { return hb::rnn_impl(); }

int hb_vec_scale(float* x, float s, int n, void* stream) {
  HB_CHECK_ARG(x && n > 0, "bad argument");
  return hb::launch_vec_scale(x, s, n, (cudaStream_t)stream);
}
}
