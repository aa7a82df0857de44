/*
 * harl_b200 -- C ABI of the B200-native HAPPO/HATRPO on-policy hot path.
 *
 * The reference (PKU-MARL/HARL @ d539bad2) is pure Python/PyTorch and has NO FFI; the
 * boundary it exposes for this path is the duck-typed Python plugin surface
 * (RUNNER_REGISTRY / ALGO_REGISTRY / buffer classes, SURVEY.md section 8(b)).  This header
 * is the C-ABI a maintainer would bind (ctypes, see INTEGRATION.md) from those Python
 * classes: every entry point below names the reference function it replaces.
 *
 * Conventions
 *   - plain C types only: raw device pointers, sizes, POD structs; no torch types.
 *   - every function returns 0 on success, <0 (hb_status) on error; the message is in
 *     hb_last_error() (thread-local).  No exceptions / exit() cross the ABI.
 *   - every call is asynchronous and ordered on `stream` (a cudaStream_t passed as void*);
 *     no call synchronises the device.
 *   - the caller owns every buffer; scratch comes from a caller-allocated workspace sized
 *     by hb_workspace_bytes().  The library keeps no device allocation of its own.
 *   - all tensors are fp32, row-major, contiguous unless a leading dimension is given.
 *   - unsupported configurations return HB_ERR_UNSUPPORTED (Python raises
 *     NotImplementedError): there is no CPU fallback.
 */
#ifndef HARL_B200_H
#define HARL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HB_VERSION 100
#define HB_MAX_LAYERS 4
#define HB_MAX_AGENTS 32
#define HB_MAX_TENSORS 40

typedef enum hb_status {
  HB_OK = 0,
  HB_ERR_INVALID = -1,     /* bad argument (null pointer, negative size, ...) */
  HB_ERR_UNSUPPORTED = -2, /* configuration outside the implemented path (no CPU fallback) */
  HB_ERR_WORKSPACE = -3,   /* workspace too small */
  HB_ERR_CUDA = -4         /* CUDA runtime error (launch failure, ...) */
} hb_status;

typedef enum hb_activation { /* harl/utils/models_tools.py:28-50 get_active_func */
  HB_ACT_RELU = 0,
  HB_ACT_TANH = 1,
  HB_ACT_SIGMOID = 2,
  HB_ACT_LEAKY_RELU = 3,
  HB_ACT_SELU = 4,
  HB_ACT_HARDSWISH = 5,
  HB_ACT_IDENTITY = 6
} hb_activation;

typedef enum hb_head {
  HB_HEAD_DISCRETE = 0, /* Categorical, harl/models/base/distributions.py:37-55 */
  HB_HEAD_BOX = 1,      /* DiagGaussian, distributions.py:58-89 */
  HB_HEAD_VALUE = 2     /* v_out Linear(h,1), harl/models/value_function_models/v_net.py:41-44 */
} hb_head;

/* One actor (StochasticPolicy, stochastic_policy.py:12-53) or critic (VNet, v_net.py:10-46):
 * [LN(in)] -> [Linear -> act -> LN] x n_layers -> [GRU x rnn_layers -> LN] -> head. */
typedef struct hb_net_desc {
  int32_t in_dim;               /* obs / share-obs dim */
  int32_t n_layers;             /* len(hidden_sizes), 1..HB_MAX_LAYERS */
  int32_t hidden[HB_MAX_LAYERS];/* hidden_sizes; each a multiple of 4, <= 256 */
  int32_t feature_norm;         /* model.use_feature_normalization */
  int32_t activation;           /* hb_activation */
  int32_t rnn_layers;           /* 0 = MLP, else model.recurrent_n */
  int32_t head;                 /* hb_head */
  int32_t out_dim;              /* n actions (Discrete), act_dim (Box), 1 (value) */
  float std_x_coef;             /* model.std_x_coef (Box) */
  float std_y_coef;             /* model.std_y_coef (Box) */
} hb_net_desc;

/* Flat parameter layout: tensors in the reference state_dict order, each start aligned to
 * 4 floats.  names[i] is the reference state_dict key. */
typedef struct hb_net_layout {
  int32_t n_tensors;
  int32_t total;                       /* floats, including alignment padding */
  int32_t offset[HB_MAX_TENSORS];
  int32_t rows[HB_MAX_TENSORS];        /* 2-D tensors: [rows, cols]; 1-D: rows = 1 */
  int32_t cols[HB_MAX_TENSORS];
  char names[HB_MAX_TENSORS][48];
  int32_t prepared_total;              /* floats of the derived ("prepared") weight buffer */
} hb_net_layout;

/* ---- library ------------------------------------------------------------------------ */
int hb_version(void);
const char* hb_last_error(void);
/* Asynchronous-error probe: cudaGetLastError on the calling thread (no sync). */
int hb_sync_check(void);

/* Number of CUDA kernels this library has launched in this process (bench.py's gpu_launches). */
uint64_t hb_kernel_launch_count(void);
/* Per-kernel timing for the roofline pass: after hb_profile_begin an event is recorded on the
 * launching stream after every kernel; hb_profile_end synchronises and writes "label count total_ms"
 * lines (sorted by time) into out, returning the byte count. */
int hb_profile_begin(void* stream);
int hb_profile_end(char* out, int out_size);

/* GEMM implementation of the MLP blocks: 0 = FP32 SIMT, 1 = tcgen05 tensor cores with the error-compensated
 * 3xTF32 split (fp32-level accuracy; default); any other value returns HB_ERR_INVALID.  Call hb_net_prepare after
 * changing it (the tensor-core path reads pre-packed operand images from the prepared buffer). */
int hb_set_gemm_impl(int impl);
int hb_get_gemm_impl(void);

/* Fused update kernel (one persistent tcgen05 launch per update: feature norm -> MLP -> head -> loss -> backward, activations
 * never leave the SM; fp16 hi/lo split operands with fp32 accumulation): 1 = use it for the shapes it covers (MLP nets with
 * two equal hidden layers of 32 / 64 / 128 units, feature normalisation, in_dim <= 64, out_dim <= 16; default), 0 = always the
 * layer-wise kernels.  Env HB_FUSED=0 selects 0.  hb_set_gemm_impl(0) (FP32 SIMT) also disables it. */
int hb_set_fused_update(int on);
int hb_get_fused_update(void);
/* Profiling aid: per-CTA, per-phase SM-clock cycle totals of the fused kernel (thread 64 of every CTA).  enable(1) clears and
 * arms the table; read synchronises the device and copies [148][16] uint64 (slots: fused_update.cu PhaseClock laps). */
int hb_fused_timing_enable(int on);
int hb_fused_timing_read(unsigned long long* out);

/* ---- network parameter plumbing ------------------------------------------------------ */
int hb_net_layout_of(const hb_net_desc* d, hb_net_layout* out);
/* Derived weights the kernels read (transposed Linear weights, feature-norm affine folded
 * into layer 1).  Must be re-run after every parameter change; hb_clip_adam_step does so. */
int hb_net_prepare(const hb_net_desc* d, const float* params, float* prepared, void* stream);
/* Scratch needed for `rows` rows.  mode: 0 = inference/evaluate (forward only), 1 = gradient. */
size_t hb_workspace_bytes(const hb_net_desc* d, int64_t rows, int mode);

/* ---- rollout side ------------------------------------------------------------------- */
/* OnPolicyBaseRunner.insert mask derivation, harl/runners/on_policy_base_runner.py:358-433.
 * dones [N,A] u8, bad_transition [N,A] u8.  Writes, for every agent a, masks_next[a][N],
 * active_next[a][N]; critic masks [N] (EP) / [N,A] (FP) and bad_masks likewise; zeroes the
 * rows of finished envs in the given rnn-state slots (nullable tables / pointers are skipped). */
typedef struct hb_insert_args {
  int32_t n_envs, n_agents, state_type_fp;
  int32_t actor_rnn_row, critic_rnn_row;      /* floats per env row (R*h); 0 = none */
  const uint8_t* dones;
  const uint8_t* bad_transition;
  float* actor_masks_next[HB_MAX_AGENTS];
  float* actor_active_next[HB_MAX_AGENTS];
  float* actor_rnn_next[HB_MAX_AGENTS];
  float* critic_masks_next;
  float* critic_bad_next;
  float* critic_rnn_next;
  /* optional episode-return bookkeeping of the logger (harl/common/base_logger.py:52-65), device-side:
   * ep_return[n] += mean_a rewards[n,a]; when env n finishes: done_sum += (ep_return[n], 1), ep_return[n] = 0. */
  const float* rewards;            /* element (n,a) at rewards[n*reward_stride_n + a*reward_stride_a]; NULL = off */
  int64_t reward_stride_n, reward_stride_a;
  float* ep_return;                /* [n_envs] */
  double* done_sum;                /* [2] */
} hb_insert_args;
int hb_rollout_insert_masks(const hb_insert_args* a, void* stream);

/* StochasticPolicy.forward (get_actions / act), stochastic_policy.py:55-91 + act.py:44-80.
 * Samples with Philox4x32-10 keyed by (seed, offset, row); deterministic=1 takes the mode.
 * actions [rows, ad] (Discrete: ad=1, the index as float), logp [rows, ad]. */
int hb_policy_act(const hb_net_desc* d, const float* prepared, const float* obs, int64_t rows,
                  const float* avail, int deterministic, uint64_t seed, uint64_t offset,
                  float* actions, float* logp, void* ws, size_t ws_bytes, void* stream);

/* One rollout step of OnPolicyBaseRunner.collect (on_policy_base_runner.py:285-340): get_actions for every agent
 * and get_values for the critic in one call, each written straight into its rollout-buffer slot. */
typedef struct hb_collect_args {
  int32_t n_agents, deterministic;
  int64_t rows;                                  /* rollout threads */
  uint64_t offset;                               /* Philox stream offset of this step */
  const hb_net_desc* actor_desc[HB_MAX_AGENTS];
  const float* actor_prepared[HB_MAX_AGENTS];
  const float* obs[HB_MAX_AGENTS];               /* [rows, in_dim_a] */
  const float* avail[HB_MAX_AGENTS];             /* [rows, n_act] or NULL */
  float* actions[HB_MAX_AGENTS];                 /* [rows, ad] */
  float* logp[HB_MAX_AGENTS];                    /* [rows, ad] */
  uint64_t seed[HB_MAX_AGENTS];
  const hb_net_desc* critic_desc;                /* NULL = skip the critic */
  const float* critic_prepared;
  const float* share_obs;                        /* [critic_rows, sd] */
  int64_t critic_rows;                           /* rows (EP) or rows * n_agents (FP) */
  float* values;                                 /* [critic_rows, 1] */
  const uint64_t* offset_base;                   /* device counter added to `offset` inside the kernel, or NULL:
                                                    lets a CUDA graph of T rollout steps be replayed with fresh
                                                    random streams (see hb_counter_add) */
  /* recurrent (GRU) nets only: this step's hidden-state / mask slots and where the new states go (normally the next
   * slot; hb_rollout_insert_masks then zeroes the rows of finished envs).  With any recurrent net the step runs the
   * per-net kernels (trunk, GRU cell, head) instead of the single fused launch. */
  const float* actor_rnn[HB_MAX_AGENTS];         /* [rows, recurrent_n * h] */
  float* actor_rnn_out[HB_MAX_AGENTS];
  const float* actor_masks[HB_MAX_AGENTS];       /* [rows] */
  const float* critic_rnn;                       /* [critic_rows, recurrent_n * h] */
  float* critic_rnn_out;
  const float* critic_masks;                     /* [critic_rows] */
} hb_collect_args;
int hb_rollout_collect(const hb_collect_args* a, void* ws, size_t ws_bytes, void* stream);
/* *counter += inc on the device (one thread).  Stream-ordered; capturable into a CUDA graph. */
int hb_counter_add(uint64_t* counter, uint64_t inc, void* stream);

/* VNet.forward (VCritic.get_values), v_net.py:48-67. values [rows,1]. */
int hb_value_forward(const hb_net_desc* d, const float* prepared, const float* cent_obs,
                     int64_t rows, float* values, void* ws, size_t ws_bytes, void* stream);

/* ---- returns / advantages ----------------------------------------------------------- */
/* OnPolicyCriticBuffer{EP,FP}.compute_returns, on_policy_critic_buffer_ep.py:97-200, fused
 * with the advantage computation of on_policy_ha_runner.py:26-33.
 * rewards [T,C], value_preds/masks/bad_masks/returns [T+1,C] (C = N or N*A), next_value [C].
 * vn_state: device float[3] = (running_mean, running_mean_sq, debiasing_term) or NULL.
 * advantages [T,C] nullable.  Bit-exact with the reference (separately rounded mul/add). */
int hb_gae_returns(const float* rewards, float* value_preds, const float* masks,
                   const float* bad_masks, const float* next_value, float* returns,
                   float* advantages, int32_t T, int64_t C, float gamma, float gamma_lambda,
                   int use_gae, int use_proper_time_limits, const float* vn_state, void* stream);

/* One launch copying n <= HB_COPY_MAX_SEGS contiguous device segments (16-byte aligned starts, sizes in whole 4-byte
 * words): an env's per-step outputs into their rollout-buffer slots -- what OnPolicyBaseRunner.insert
 * (harl/runners/on_policy_base_runner.py:340-415) does with one NumPy assignment per array. */
#define HB_COPY_MAX_SEGS 16
typedef struct hb_copy_seg {
  void* dst;
  const void* src;
  int64_t bytes;
} hb_copy_seg;
int hb_copy_segments(const hb_copy_seg* segs, int32_t n, void* stream);

/* ---- multi-GPU exchange (SURVEY.md section 8(e)): one-shot sum-allreduce of a small bucket over NVLink peer memory.
 * The reference is single-process; what is exchanged is the part of its batch means that lives on other GPUs when the
 * rollout threads are sharded: the flat gradient of one optimiser step (happo.py:85-97, v_critic.py:116-140) and the
 * loss / advantage / ValueNorm normalisers (happo.py:74-91, on_policy_ha_runner.py:38-47, valuenorm.py:47-64).
 *
 * hb_comm_create allocates this rank's exchange region on the current device (2 slots of slot_bytes + flags) and writes
 * its 64-byte CUDA IPC handle to ipc_handle_out64; the caller gathers the handles of all ranks (any transport) and
 * passes the world x 64 bytes, in rank order, to hb_comm_open_peers.  hb_allreduce_bucket sums buf[0..n) (dtype 0 =
 * float32, 1 = float64) over the ranks IN RANK ORDER, in place, on `stream`: every rank obtains the bit-identical
 * result.  All ranks must issue the same sequence of calls on a communicator; use one communicator per stream.
 * hb_comm_status: 0, or 1 + r if rank r did not arrive within HB_COMM_TIMEOUT_S (default 20 s) in some exchange. */
int hb_comm_create(int32_t rank, int32_t world, size_t slot_bytes, void** comm_out, void* ipc_handle_out64);
int hb_comm_open_peers(void* comm, const void* all_handles);
int hb_allreduce_bucket(void* comm, void* buf, int64_t n, int32_t dtype, void* stream);
int hb_comm_status(void* comm);
int hb_comm_destroy(void* comm);

/* How the time-segmented GAE kernel (T <= 256) carries the running GAE between its segments: 1 = sequentially
 * (default; bit-identical to the reference's on_policy_critic_buffer_ep.py:111-140 loop), 2 = by a parallel affine scan
 * (advantages within 1e-6 of max|adv| of the sequential result); any other value returns HB_ERR_INVALID.  Longer
 * rollouts and the return branch without GAE always run the bit-exact column-tile kernel.  Env HB_GAE_IMPL=2 selects 2
 * at start-up; any other value gives 1. */
int hb_set_gae_impl(int impl);
int hb_get_gae_impl(void);

/* Masked moments for happo.py:122-127 / on_policy_ha_runner.py:36-45:
 * out3 (device double[3]) += (sum x*w, sum x*x*w, sum w) with w = (weight != 0) or 1. */
int hb_masked_moments(const float* x, const float* weight, int64_t n, double* out3, void* stream);
/* x_out = (x - mean) / (std + 1e-5) from moments3 (population std). */
int hb_normalize_by_moments(const float* x, float* x_out, int64_t n, const double* moments3,
                            void* stream);

/* ValueNorm.update, harl/common/valuenorm.py:47-64, from moments3 = (sum, sumsq, count). */
int hb_valuenorm_update(float* vn_state, const double* moments3, double beta, void* stream);
/* ValueNorm.normalize / denormalize, valuenorm.py:66-92 (elementwise). */
int hb_valuenorm_apply(const float* vn_state, const float* x, float* y, int64_t n,
                       int denormalize, void* stream);

/* ---- sequential-agent update -------------------------------------------------------- */
typedef struct hb_ppo_hyper {  /* harl/configs/algos_cfgs/happo.yaml algo.* */
  float clip_param;
  float entropy_coef;
  int32_t use_policy_active_masks;
  int32_t action_aggregation_prod;  /* 1 = prod, 0 = mean */
  int32_t use_clip;                 /* 1 = HAPPO, 0 = HAA2C (no clipping) */
} hb_ppo_hyper;

/* Buffer-resident batch for one actor.  `index` (nullable) maps batch row -> buffer row
 * (time-major flat index t*N+n, Appendix D of SURVEY.md); NULL = identity. */
typedef struct hb_actor_batch {
  const float* obs;          /* [R, in_dim] */
  const float* actions;      /* [R, ad] */
  const float* old_logp;     /* [R, ad] */
  const float* adv;          /* [R] */
  const float* factor;       /* [R] or NULL (= 1) */
  const float* active;       /* [R] */
  const float* avail;        /* [R, n_act] or NULL */
  const int32_t* index;      /* [rows] or NULL */
  int64_t rows;
  /* recurrent policies only (RNNLayer sequence branch, rnn.py:33-78; generators of Appendix D): the batch is
   * seq_len steps x (rows / seq_len) sequences, rows step-major (row = s * B + j).  rnn_states is the buffer's
   * [R, recurrent_n * h] array: sequence j starts from buffer row (index ? index[j] : j); masks [R] multiplies
   * the state before every step. */
  const float* rnn_states;
  const float* masks;
  int64_t seq_len;
} hb_actor_batch;

/* StochasticPolicy.evaluate_actions over buffer rows (the old/new log-prob sweeps of
 * on_policy_ha_runner.py:66-113).  logp_out [rows, ad].  If factor_inout != NULL also applies
 * on_policy_ha_runner.py:116-124:  factor *= agg_d exp(logp_new - logp_ref[rows, ad]). */
int hb_policy_evaluate(const hb_net_desc* d, const float* prepared, const hb_actor_batch* b,
                       float* logp_out, const float* logp_ref, float* factor_inout,
                       int action_aggregation_prod, void* ws, size_t ws_bytes, void* stream);

/* HAPPO.update forward + loss + backward, harl/algorithms/actors/happo.py:28-91.
 * grad (layout of hb_net_layout, zeroed inside) receives d(policy_loss - entropy_coef*H)/dparams.
 * norm3: device double[3]; norm3[2] = sum(active) over the WHOLE minibatch (all ranks) if
 * use_policy_active_masks else the row count -- the caller reduces it before the call.
 * scalars (device double[4]) += (sum -factor*min(s1,s2)*w, sum entropy*w, sum ratio, rows). */
int hb_ppo_actor_grad(const hb_net_desc* d, const float* params, const float* prepared,
                      const hb_actor_batch* b, const hb_ppo_hyper* h, const double* norm3,
                      float* grad, double* scalars, void* ws, size_t ws_bytes, void* stream);

/* hb_ppo_actor_grad that also writes the log-probabilities of the batch actions under the weights it differentiates
 * (logp_out [rows, ad], identity batches only; NULL = plain hb_ppo_actor_grad).  The sequential update needs exactly
 * these numbers for the agent it is about to train -- on_policy_ha_runner.py:66-83 evaluates the whole buffer with the
 * pre-update weights, which are the weights of the first PPO epoch -- so the forward of that epoch serves both. */
int hb_ppo_actor_grad_logp(const hb_net_desc* d, const float* params, const float* prepared, const hb_actor_batch* b,
                           const hb_ppo_hyper* h, const double* norm3, float* grad, double* scalars, float* logp_out,
                           void* ws, size_t ws_bytes, void* stream);

typedef struct hb_value_hyper { /* happo.yaml algo.*: VCritic, v_critic.py:24-37 */
  float clip_param;
  float huber_delta;
  float value_loss_coef;
  int32_t use_huber_loss;
  int32_t use_clipped_value_loss;
} hb_value_hyper;

typedef struct hb_critic_batch {
  const float* share_obs;    /* [R, in_dim] */
  const float* value_preds;  /* [R] */
  const float* returns;      /* [R] */
  const int32_t* index;      /* nullable */
  int64_t rows;
  const float* rnn_states;   /* recurrent critics: as in hb_actor_batch */
  const float* masks;
  int64_t seq_len;
} hb_critic_batch;

/* VCritic.update forward + cal_value_loss + backward, v_critic.py:75-146.
 * vn_state nullable (already updated with this batch, v_critic.py:90-95).
 * inv_count = 1 / (global number of rows in the minibatch).
 * scalars (device double[4]) += (sum value_loss_elem, rows, 0, 0). */
int hb_value_grad(const hb_net_desc* d, const float* params, const float* prepared,
                  const hb_critic_batch* b, const hb_value_hyper* h, const float* vn_state,
                  double inv_count, float* grad, double* scalars, void* ws, size_t ws_bytes,
                  void* stream);

/* clip_grad_norm_ (happo.py:93-98) + torch.optim.Adam step (on_policy_base.py:37-42), then
 * hb_net_prepare.  grad_norm_out: device float[1] (pre-clip total norm). */
typedef struct hb_adam_hyper {
  float lr, beta1, beta2, eps, weight_decay, max_grad_norm;
  int32_t use_max_grad_norm;
  int32_t step;              /* 1-based Adam step count of this update */
} hb_adam_hyper;
int hb_clip_adam_step(const hb_net_desc* d, float* params, const float* grad, float* exp_avg,
                      float* exp_avg_sq, float* prepared, const hb_adam_hyper* h,
                      float* grad_norm_out, void* stream);

/* ---- recurrent (GRU) networks: one rollout step, rnn.py:24-32 ------------------------------------------ *
 * rnn_states [rows, recurrent_n * h] and masks [rows] are the buffer slot of this step; the new hidden state goes
 * to rnn_states_out [rows, recurrent_n * h] (StochasticPolicy.forward / VNet.forward return value).
 * offset_base (nullable): device counter added to `offset` inside the sampling kernel, as in hb_collect_args. */
int hb_policy_act_rnn(const hb_net_desc* d, const float* prepared, const float* obs, int64_t rows,
                      const float* avail, const float* rnn_states, const float* masks, int deterministic,
                      uint64_t seed, uint64_t offset, const uint64_t* offset_base, float* actions, float* logp,
                      float* rnn_states_out, void* ws, size_t ws_bytes, void* stream);
int hb_value_forward_rnn(const hb_net_desc* d, const float* prepared, const float* cent_obs, int64_t rows,
                         const float* rnn_states, const float* masks, float* values, float* rnn_states_out,
                         void* ws, size_t ws_bytes, void* stream);

/* GRU recurrence implementation: 0 = one GEMM + one gate kernel per step, 1 = persistent per-sequence kernel (h = 64; other
 * widths run per step).  Default 1 since round 2 (bit-identical to 0 on a B200: tests/test_gpu_rnn.py).
 * Env: HB_RNN_IMPL=per_step selects 0. */
int hb_set_rnn_impl(int impl);
int hb_get_rnn_impl(void);
/* Tangent block of the trust-region Fisher-vector product: 0 = FP32 FFMA tiles, 1 = tcgen05 kernel (K-doubled product,
 * LayerNorm-tangent epilogue; needs the tensor-core GEMM mode).  Default 1 since round 2 (verified against 0 on a B200:
 * tests/test_gpu_zz_wide_heads.py).  Env: HB_TRPO_JVP_IMPL=0 selects 0. */
int hb_set_trpo_jvp_impl(int impl);
int hb_get_trpo_jvp_impl(void);

/* ---- trust-region (HATRPO) update: harl/algorithms/actors/hatrpo.py:37-194, harl/utils/trpo_util.py ------- *
 * The surrogate gradient is hb_ppo_actor_grad with use_clip = 0 and entropy_coef = 0 (it returns the gradient of
 * -loss; hb_vec_scale flips the sign).  The parameter-space vectors below (v, out, x, r, p, g, full_step,
 * params0) all use the flat hb_net_layout with zero padding words. */

/* workspace for hb_trpo_fvp (covers hb_trpo_old_dist / hb_trpo_eval too) */
size_t hb_trpo_workspace_bytes(const hb_net_desc* d, int64_t rows);

/* Distribution of the CURRENT parameters per batch row -> old_dist [rows, out_dim]: torch Categorical.logits
 * (normalised) for Discrete, the mean for Box.  Replaces the no-grad old_actor.evaluate_actions of
 * trpo_util.py:79-82 (the old policy is evaluated once, not once per KL call). */
int hb_trpo_old_dist(const hb_net_desc* d, const float* prepared, const hb_actor_batch* b, float* old_dist,
                     void* ws, size_t ws_bytes, void* stream);

/* fisher_vector_product (trpo_util.py:136-158) WITHOUT the + 0.1 p term: out = d2 mean_rows KL(pi || pi) / dtheta2 . v
 * as J^T H J v (tangent pass, H / rows, backward pass), partial over this rank's rows; inv_rows = 1 / global rows.
 * The caller sum-reduces `out` over ranks, then calls hb_trpo_fvp_finish.
 * reuse_forward = 1: the previous call on this workspace was hb_trpo_fvp with the same net, parameters and batch
 * (the 11 products of one update) and nothing else used the workspace since -- the forward activations (and the
 * GRU's saved gates) are taken from it instead of being recomputed (single-chunk batches only; ignored otherwise). */
int hb_trpo_fvp(const hb_net_desc* d, const float* params, const float* prepared, const hb_actor_batch* b,
                const float* old_dist, const float* v, double inv_rows, int reuse_forward, float* out, void* ws,
                size_t ws_bytes, void* stream);
/* out += damping * v (trpo_util.py:158), plus the DiagGaussian log_std block of the Hessian (row-independent). */
int hb_trpo_fvp_finish(const hb_net_desc* d, const float* params, const float* v, float* out, float damping,
                       void* stream);

/* One backtracking-line-search trial (hatrpo.py:142-181): `prepared` holds the candidate parameters.
 * scalars (device double[4]) += (sum ratio*factor*adv*w, sum entropy*w, sum ratio, sum KL(old || new)) over rows;
 * w = active if use_policy_active_masks else 1.  params_old: flat parameters before the step (Box: old log_std). */
int hb_trpo_eval(const hb_net_desc* d, const float* prepared, const hb_actor_batch* b, const hb_ppo_hyper* h,
                 const float* old_dist, const float* params_old, double* scalars, void* ws, size_t ws_bytes,
                 void* stream);

/* conjugate_gradient (trpo_util.py:100-133) with the state on the device: cg_state = {rdotr, done}.
 * cg_init: x = 0, r = p = b.  cg_step consumes avp = (F + 0.1 I) p and is a no-op once rdotr < residual_tol. */
int hb_trpo_cg_init(const float* b, float* x, float* r, float* p, float* cg_state, int n, void* stream);
int hb_trpo_cg_step(float* p, const float* avp, float* x, float* r, float* cg_state, int n, float residual_tol,
                    void* stream);
/* hatrpo.py:123-133: shs = 0.5 x.Fx; step_size = 1/sqrt(shs/kl_threshold); full_step = step_size * x;
 * out3 (device double[3]) = (shs, step_size, expected_improve = g.full_step). */
int hb_trpo_full_step(const float* x, const float* fx, const float* g, float kl_threshold, float* full_step,
                      double* out3, int n, void* stream);
/* update_model(actor, params + fraction * full_step), hatrpo.py:143-144 (follow with hb_net_prepare). */
int hb_trpo_apply_step(float* params, const float* params0, const float* full_step, float fraction, int n,
                       void* stream);
int hb_vec_scale(float* x, float s, int n, void* stream);

/* ---- batched MPE simple_spread environment (SURVEY.md section 8(f) row 1) --------------------------------------- *
 * Replaces, for `pettingzoo_mpe` / `simple_spread_v2`, the per-env PettingZooMPEEnv.step + ShareSubprocVecEnv of
 * harl/envs/pettingzoo_mpe/pettingzoo_mpe_env.py:41-88 and harl/envs/env_wrappers.py by ONE launch over all rollout
 * threads that writes the next observations / state / team reward / done flags straight into the rollout-buffer slots.
 * World state (device, owned by the caller): pos, vel [n_envs, n_agents, 2], landmarks [n_envs, n_landmarks, 2],
 * step_count [n_envs] int32, episode [n_envs] uint64.  reset_all = 1: (re)initialise every world (episode 0) and
 * write observations / state only.  Initial positions: Philox4x32-10 keyed by (seed, env, episode). */
#define HB_MPE_MAX_AGENTS 8
typedef struct hb_mpe_args {
  int32_t n_envs, n_agents, n_landmarks;
  int32_t continuous;        /* 0: Discrete(5) action index as float [n_envs, 1]; 1: Box(5) [n_envs, 5] */
  int32_t max_cycles;        /* truncation length (25), pettingzoo_mpe_env.py:22-27 */
  int32_t reset_all;
  uint64_t seed;
  float* pos; float* vel; float* landmarks;
  int32_t* step_count; uint64_t* episode;
  const float* actions[HB_MPE_MAX_AGENTS];
  float* obs_out[HB_MPE_MAX_AGENTS];   /* [n_envs, 4 + 2 n_landmarks + 4 (n_agents - 1)] per agent */
  float* share_obs_out;                /* [n_envs, n_agents * obs_dim] (EP state), nullable */
  float* rewards_out;                  /* [n_envs] team reward, nullable */
  float* rewards_na_out;               /* [n_envs, n_agents], nullable */
  uint8_t* dones_out; uint8_t* bad_out;/* [n_envs, n_agents], nullable */
} hb_mpe_args;
int hb_mpe_spread_step(const hb_mpe_args* a, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HARL_B200_H */
