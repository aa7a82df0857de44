"""Benchmark of the HAPPO on-policy hot path (BASELINE.json metric: env-steps/sec, whole box).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload C2]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W     (N > 1)

One "step" = one full training iteration of the runner on synthetic tensors of the workload's
shapes: T x (collect -> env.step -> insert) -> GAE -> sequential-agent HAPPO update -> critic update
-> after_update.  value = T * N_global / seconds per iteration, the reference's own FPS formula
(harl/common/base_logger.py:70-87; agents do not multiply the count).  Weak scaling: every GPU
keeps the workload's n_rollout_threads, so N_global = N * n_rollout_threads.

Rank 0 prints ONE JSON line.  Extra objects (see DESIGN.md "Measurement"):
  roofline      dominant kernel of the step, timed live with CUDA events on the launching stream
  cpu_baseline  the UNMODIFIED reference (baseline/_ref, driven by baseline/ref_runner.py) on this box's host cores, on a
                256-thread sample of the workload (N=1 only)
  e2e           same metric with the env on the HOST: pinned H2D of every env output and D2H of the
                actions each rollout step, plus the D2H of the train infos, inside the timed region
--impl reference times the unmodified reference's own OnPolicyHARunner.run() (baseline/_ref travels with the snapshot) at
the bench configuration itself, >= 3 timed iterations within --ref-budget-s; --ref-cuda sets its device.cuda = True;
--ref-cross-check adds the oracle CPU port (oracle/runner.py) as a cross-check.  --scaling strong splits the workload's
n_rollout_threads over the ranks instead of giving each rank all of them.
--dump-outputs DIR writes what the last timed iteration computed as DIR/<name>.npy (see dump_outputs), so that two
builds run with the same arguments -- hence the same seeded inputs -- can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs (SURVEY.md section 8(d)).  C2 is the configuration the metric is quoted on.
WORKLOADS = {
    "C1": dict(desc="HAPPO pettingzoo_mpe simple_spread_v2 3 agents n_rollout_threads=8 (synthetic tensors)",
               env="pettingzoo_mpe", env_args=dict(scenario="simple_spread_v2", continuous_actions=False), n=8, T=200,
               hidden=[128, 128], algo={}),
    "C2": dict(desc="HAPPO synthetic-MPE obs_dim=18 act_dim=5 3 agents n_rollout_threads=4096 T=200",
               env="pettingzoo_mpe", env_args=dict(scenario="simple_spread_v2", continuous_actions=False), n=4096, T=200,
               hidden=[128, 128], algo={}),
    "C3": dict(desc="HAPPO MAMuJoCo HalfCheetah-v2 6x1 continuous n_rollout_threads=1024 T=200",
               env="mamujoco", env_args=dict(scenario="HalfCheetah-v2", agent_conf="6x1"), n=1024, T=200,
               hidden=[128, 128, 128], algo=dict(clip_param=0.05, ppo_epoch=15, critic_epoch=15)),
    "C5": dict(desc="HAPPO MAMuJoCo Humanoid-v2 17x1 n_rollout_threads=1024 per GPU T=200",
               env="mamujoco", env_args=dict(scenario="Humanoid-v2", agent_conf="17x1"), n=1024, T=200,
               hidden=[128, 128, 128], algo=dict(clip_param=0.1, entropy_coef=0.0)),
    # C1 on the learnable task itself: the batched CUDA simple_spread env (harl_b200/envs/mpe_spread.py), tuned N = 20
    "C1M": dict(desc="HAPPO pettingzoo_mpe simple_spread_v2 3 agents n_rollout_threads=20, native batched env (tuned config)",
                env="pettingzoo_mpe", env_args=dict(scenario="simple_spread_v2", continuous_actions=False, backend="native"), n=20,
                T=200, hidden=[128, 128], algo={}),
    # BASELINE.json's C4 and its two halves: the trust-region update at C2 shapes (C2T), GRU policies / FP critic at the
    # synthetic-SMAC shapes under HAPPO (C4R).  Secondary workloads (--workload), run with --no-cpu-baseline --no-e2e.
    "C2T": dict(desc="HATRPO synthetic-MPE obs_dim=18 act_dim=5 3 agents n_rollout_threads=4096 T=200",
                env="pettingzoo_mpe", env_args=dict(scenario="simple_spread_v2", continuous_actions=False), n=4096, T=200,
                hidden=[128, 128], algo={}, algo_name="hatrpo"),
    "C4": dict(desc="HATRPO synthetic-SMAC 5 agents obs_dim=128 Discrete(12) n_rollout_threads=2048 T=160 GRU chunk 10, FP critic "
                    "(BASELINE.json configs[3], one GPU's worth)",
               env="smac", env_args=dict(map_name="5m_vs_6m"), n=2048, T=160, hidden=[64, 64, 64], algo=dict(gamma=0.95),
               model=dict(use_recurrent_policy=True, data_chunk_length=10), algo_name="hatrpo"),
    "C4R": dict(desc="HAPPO synthetic-SMAC 5 agents obs_dim=128 Discrete(12) n_rollout_threads=2048 T=160 GRU chunk 10, FP critic",
                env="smac", env_args=dict(map_name="5m_vs_6m"), n=2048, T=160, hidden=[64, 64, 64], algo=dict(gamma=0.95),
                model=dict(use_recurrent_policy=True, data_chunk_length=10)),
}


STRONG = False   # --scaling strong: the workload's n_rollout_threads is the GLOBAL count


def make_args(wl, world, host_env=False, n_override=None):
    from harl_b200.utils.configs_tools import get_defaults_yaml_args

    w = WORKLOADS[wl]
    algo_args, env_args = get_defaults_yaml_args(w.get("algo_name", "happo"), w["env"])
    env_args.update(w["env_args"])
    env_args["host"] = host_env
    n = n_override or w["n"]
    algo_args["train"].update(n_rollout_threads=n * (1 if STRONG else world), episode_length=w["T"], num_env_steps=10**12,
                              log_interval=10**9, eval_interval=10**9)
    algo_args["eval"]["use_eval"] = False
    algo_args["model"]["hidden_sizes"] = list(w["hidden"])
    algo_args["algo"].update(w["algo"])
    algo_args["model"].update(w.get("model", {}))
    algo_args["logger"]["log_dir"] = tempfile.mkdtemp(prefix="harl_b200_bench_")
    args = dict(algo=w.get("algo_name", "happo"), env=w["env"], exp_name="bench", load_config="")
    return args, algo_args, env_args


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


def timed_iterations(runner, steps, warmup, torch, dist_on, sample_clocks=False):
    """W untimed + K timed iterations, CUDA events, barrier + synchronize on both sides, max over ranks."""
    ep = getattr(runner, "_bench_episode", 0)
    for _ in range(warmup):
        ep += 1
        runner.run_iteration(ep, 10**9)
    if dist_on:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    sampler = None
    if sample_clocks:
        sampler = ClockSampler(torch.cuda.current_device())
        sampler.start()
    from harl_b200 import _lib as L

    l0 = L.lib.hb_kernel_launch_count()
    g0 = getattr(runner, "graph_replayed_launches", 0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        ep += 1
        runner.run_iteration(ep, 10**9)
    ev1.record()
    torch.cuda.synchronize()
    # library kernels launched directly + those replayed from the captured rollout graph
    launches = L.lib.hb_kernel_launch_count() - l0 + getattr(runner, "graph_replayed_launches", 0) - g0
    if dist_on:
        torch.distributed.barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device="cuda")
    if dist_on:
        torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
    runner._bench_episode = ep
    return ms.item(), launches, (sampler.summary() if sampler else None)


DUMP_ROWS = 16384   # rollout rows (t, thread) of the seeded sample written per buffer tensor


def dump_outputs(runner, out_dir, torch):
    """Write what the runner's last iteration handed back (rank 0's shard): the train infos of every agent and of the
    critic (float64), the flat parameters of every actor and of the critic after the update, the ValueNorm statistics,
    and a fixed, seeded sample of DUMP_ROWS rollout rows of the buffers it filled -- each agent's actions and their
    log-probs, the critic's value predictions, returns and advantages (float32).  0.9 MB at C2."""
    import numpy as np

    torch.cuda.synchronize()
    T, N = runner.algo_args["train"]["episode_length"], runner.n_local
    pick = torch.randperm(T * N, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values.to(runner.device)

    def rows(x):   # [T or T + 1, N, ...] -> the sampled rows of the first T steps
        return x[:T].reshape(T * N, *x.shape[2:]).index_select(0, pick)

    actor_infos, critic_info = runner.last_train_infos
    out = {f"actor_info_{k}": np.array([info[k] for info in actor_infos], np.float64) for k in sorted(actor_infos[0])}
    out.update({f"critic_info_{k}": np.array([critic_info[k]], np.float64) for k in sorted(critic_info)})
    for a, (actor, buf) in enumerate(zip(runner.actor, runner.actor_buffer)):
        out[f"actor{a}_params"] = actor.actor.params
        out[f"actor{a}_actions"] = rows(buf.actions)
        out[f"actor{a}_action_log_probs"] = rows(buf.action_log_probs)
    cb = runner.critic_buffer
    out["critic_params"] = runner.critic.critic.params
    for name in ("value_preds", "returns", "advantages"):
        out[f"critic_{name}"] = rows(getattr(cb, name))
    if runner.value_normalizer is not None:
        out["value_normalizer"] = torch.cat([v.reshape(-1).double() for v in runner.value_normalizer.state_dict().values()])
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        if torch.is_tensor(v):
            v = v.detach().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), v if v.dtype == np.float64 else v.astype(np.float32))


def kernel_profile(runner, torch):
    """One extra iteration with an event after every kernel launch -> [(label, count, total_ms)]."""
    from harl_b200 import _lib as L

    torch.cuda.synchronize()
    runner.time_phases = True
    runner._bench_episode += 1
    runner.run_iteration(runner._bench_episode, 10**9)  # phase timers without per-kernel events
    runner.time_phases = False
    # Profile the update phase only: there the host runs far ahead of the device, so the gap between
    # consecutive post-launch events is the kernel's own duration.  (In the rollout the device waits for
    # Python between steps and the gaps would be charged to the kernels.)
    runner._bench_episode += 1
    runner.logger.episode_init(runner._bench_episode)
    for step in range(runner.algo_args["train"]["episode_length"]):
        values, actions, logp, rnn, rnn_c = runner.collect(step)
        obs, share_obs, rewards, dones, infos, avail = runner.envs.step(actions)
        runner.insert((obs, share_obs, rewards, dones, infos, avail, values, actions, logp, rnn, rnn_c))
    runner.compute()
    torch.cuda.synchronize()
    overlap, runner.overlap_critic_update = getattr(runner, "overlap_critic_update", True), False  # one stream: clean gaps
    runner.train()  # unprofiled pass: the critic's workspace on this stream is allocated here, not inside a gap
    torch.cuda.synchronize()
    L.call("hb_profile_begin", L.stream_ptr())
    runner.train()
    runner.overlap_critic_update = overlap
    buf = C.create_string_buffer(1 << 16)
    n = L.lib.hb_profile_end(buf, len(buf))
    runner.after_update()
    rows = []
    for line in buf.raw[:max(n, 0)].decode().strip().splitlines():
        label, cnt, ms = line.rsplit(" ", 2)
        rows.append((label, int(cnt), float(ms)))
    return rows


GEMM_LABEL = re.compile(r"^(tc_)?(linear_ln_fwd|dx_ln_bwd|dw_accum)")
FUSED_LABEL = re.compile(r"^fused_(actor_update|critic_update|evaluate)")
NET_SHAPES = {}   # filled from the runner: od, sd, na (Discrete) / ad (Box), hidden, avail


def _fused_work(label):
    """Algorithmic (bytes, FLOPs) per launch of a fused kernel, SURVEY.md section 8(d): every input element of a row is
    moved once (weights excluded); FLOPs = 2 * in * out per Linear, x3 for forward + backward."""
    m = re.match(r"(\w+)\[M(\d+),N(\d+),K(\d+)\]", label)
    name, M, H, K = m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(4))
    sh = NET_SHAPES
    out = 1 if name == "fused_critic_update" else sh.get("out", 5)
    fwd = 2.0 * (K * H + H * H + H * out)
    if name == "fused_critic_update":
        return M * 4.0 * (K + 2), M * 3.0 * fwd
    aw = 1 if sh.get("discrete", True) else sh.get("out", 1)          # stored action / log-prob width
    avail = 4.0 * sh.get("out", 5) if (sh.get("discrete", True) and sh.get("avail", True)) else 0.0
    if name == "fused_actor_update":
        return M * (4.0 * K + 4.0 * aw + 4.0 * aw + 12.0 + avail), M * 3.0 * fwd
    return M * (4.0 * K + 4.0 * aw + avail + 4.0 * aw), M * fwd        # evaluate: + the log-probs written


def _algorithmic(label):
    """(kind, amount per launch) of a profiled kernel label ``name[M..,N..,K..]`` (DESIGN.md section 5)."""
    m = re.match(r"([\w]+)\[M(\d+),N(\d+),K(\d+)\]", label)
    if not m:
        return None, None
    name, M, N, K = m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(4))
    if FUSED_LABEL.match(name):
        nbytes, flops = _fused_work(label)
        return "gemm", (flops, nbytes)
    if GEMM_LABEL.match(name):
        # algorithmic FLOPs: one fp32-accurate product (3xTF32 issues 3 MMAs for it); algorithmic bytes: every operand /
        # result row moved once -- forward reads X[M,K], writes Z and Y [M,N]; dX reads dZ[M,K'] and Z[M,N], writes dZ'[M,N];
        # dW reads dZ[M,N] and X[M,K] (weights, <= 64 KB, excluded)
        nbytes = 4.0 * M * (N + K) if "dw_accum" in name else 4.0 * M * (K + 2 * N)
        return "gemm", (2.0 * M * N * K, nbytes)
    if name.startswith("policy_head_grad"):  # features + pre-LN z + dZ out (K floats each) + stats + 5 row scalars + avail
        return "bytes", M * (12.0 * K + 8 + 20 + 4 * N)
    if name.startswith("value_head_grad"):
        return "bytes", M * (12.0 * K + 8 + 8)
    if name.startswith("policy_head") or name.startswith("value_head"):
        return "bytes", M * (4.0 * K + 8 + 4 * N)
    if name.startswith("feat_norm"):  # N = padded output width, K = input width
        return "bytes", M * 4.0 * (K + N)
    return None, None


def _rate(row, peaks):
    label, cnt, ms = row
    kind, amount = _algorithmic(label)
    sec = 1e-3 * ms / cnt
    tf_peak = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops")
    hbm_peak = peaks.get("hbm_gbs_sustained") or peaks.get("hbm_gbs")
    if kind == "gemm":
        # two roofs; the binding one is the larger time bound.  At 21-32 FLOP/B these layer-wise GEMM kernels sit far
        # below the tensor/HBM ridge (~210 FLOP/B), so HBM binds; the tensor-side numbers are kept alongside.
        flops, nbytes = amount
        tf, gbs = flops / sec / 1e12, nbytes / sec / 1e9
        t_tensor, t_hbm = flops / (tf_peak * 1e12), nbytes / (hbm_peak * 1e9)
        side = dict(flops_per_launch=flops, bytes_per_launch=nbytes, flop_per_byte=flops / nbytes,
                    tensor_tflops=tf, tensor_peak_tflops=tf_peak, frac_of_tensor_peak=tf / tf_peak,
                    hbm_gbs=gbs, hbm_peak_gbs=hbm_peak, frac_of_hbm_peak=gbs / hbm_peak)
        if FUSED_LABEL.match(label.split("[")[0]):
            # fp32-level accuracy out of the f16 pipe costs three MMAs per product (hi*hi + lo*hi + hi*lo): what the tensor
            # pipe actually issues is 3x the algorithmic FLOPs
            side.update(mma_passes_per_product=3, issued_tensor_tflops=3.0 * tf, issued_frac_of_tensor_peak=3.0 * tf / tf_peak)
        if t_hbm >= t_tensor:
            return dict(bound="hbm", achieved=gbs, peak=hbm_peak, unit="GB/s", frac=gbs / hbm_peak, **side)
        return dict(bound="tensor", achieved=tf, peak=tf_peak, unit="TFLOP/s", frac=tf / tf_peak, **side)
    if kind == "bytes":
        ach = amount / sec / 1e9
        return dict(bound="hbm", achieved=ach, peak=hbm_peak, unit="GB/s", frac=ach / hbm_peak, bytes_per_launch=amount)
    return dict(bound="hbm", achieved=None, peak=hbm_peak, unit="GB/s", frac=None)


def roofline_of(rows, peaks):
    """Roofline entry for the kernel label with the largest share of the update phase.

    GEMM kernels (the MLP layers -- tensor-pipe work by BASELINE.json's own classification) are rated in algorithmic
    FLOP/s (2MNK) against the measured dense bf16 peak; row-wise kernels in algorithmic bytes against measured HBM
    bandwidth.  ``top_gemm`` rates the largest GEMM label the same way when the top label is not a GEMM."""
    from harl_b200 import _lib as L

    total = sum(r[2] for r in rows) or 1.0
    label, cnt, ms = rows[0]
    out = {"kernel": label, "launches": cnt, "avg_us": 1e3 * ms / cnt, "share_of_update_phase": ms / total,
           "scope": "update phase (runner.train) of one iteration; phases in config.phases_ms",
           "gemm_impl": ("fused tcgen05 kernel (fp16 hi/lo split, fp32 accumulate); layer-wise fallback: " if L.lib.hb_get_fused_update() else "") +
                        {0: "fp32 SIMT", 1: "tcgen05 3xTF32", 2: "tcgen05 TF32"}[L.lib.hb_get_gemm_impl()],
           "peak_source": peaks["_source"],
           "top5": [{"kernel": r[0], "launches": r[1], "avg_us": round(1e3 * r[2] / r[1], 2), "share": round(r[2] / total, 4)}
                    for r in rows[:5]]}
    out.update(_rate(rows[0], peaks))
    gem = [r for r in rows if GEMM_LABEL.match(r[0]) or FUSED_LABEL.match(r[0])]
    if gem:
        g = dict(kernel=gem[0][0], launches=gem[0][1], avg_us=1e3 * gem[0][2] / gem[0][1], share=gem[0][2] / total)
        g.update(_rate(gem[0], peaks))
        out["top_gemm"] = g
        out["gemm_share_of_update_phase"] = sum(r[2] for r in gem) / total
    tr = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    out["traffic"] = None
    if os.path.exists(tr):
        try:
            out["traffic"] = json.load(open(tr)).get(label.split("[")[0])
        except Exception:
            pass
    return out


def gae_microbench(torch, T, C, peaks, sets=8, reps=5, impl=None):
    """hb_gae_returns alone at the workload's [T, C]: CUDA events around sets x reps launches that rotate over
    `sets` independent buffer sets (8 x 19.7 MB at C2 > the 126 MB L2, so every launch streams from HBM).
    Algorithmic bytes = 24 B per (t, column): rewards, value_preds, masks, bad_masks read; returns, advantages
    written (SURVEY section 8(d))."""
    from harl_b200 import _lib as L

    if impl is not None:   # 1 = sequential carry (default, bit-exact), 2 = parallel scan of the carry (1e-6 of max|adv|)
        prev = L.lib.hb_get_gae_impl()
        L.call("hb_set_gae_impl", impl)
        try:
            out = gae_microbench(torch, T, C, peaks, sets, reps)
        finally:
            L.call("hb_set_gae_impl", prev)
        out["kernel"] += " impl=%d (%s)" % (impl, {0: "shared-memory tiles", 1: "segmented, sequential carry", 2: "segmented, parallel scan"}[impl])
        return out
    dev = torch.device("cuda:0" if "LOCAL_RANK" not in os.environ else f"cuda:{os.environ['LOCAL_RANK']}")
    g = torch.Generator(device="cpu").manual_seed(3)
    bufs = []
    for _ in range(sets):
        rew = torch.randn(T, C, generator=g).to(dev)
        vp = torch.randn(T + 1, C, generator=g).to(dev)
        masks = (torch.rand(T + 1, C, generator=g) > 0.04).float().to(dev)
        bad = (torch.rand(T + 1, C, generator=g) > 0.02).float().to(dev)
        bufs.append((rew, vp, masks, bad, torch.randn(C, generator=g).to(dev), torch.empty(T + 1, C, device=dev),
                     torch.empty(T, C, device=dev)))
    vn = torch.tensor([0.1, 1.3, 1.0], device=dev)
    st = L.stream_ptr()

    def launch(b):
        nonlocal st
        L.call("hb_gae_returns", L.ptr(b[0]), L.ptr(b[1]), L.ptr(b[2]), L.ptr(b[3]), L.ptr(b[4]), L.ptr(b[5]), L.ptr(b[6]),
               T, C, 0.99, 0.99 * 0.95, 1, 1, L.ptr(vn), st)

    for b in bufs:
        launch(b)
    torch.cuda.synchronize()
    # the launches go through a CUDA graph: issued eagerly from Python they would be host-bound (~10 us per call)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        st = L.stream_ptr()
        for b in bufs:
            launch(b)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    # the same traffic as plain device copies (12 B read + 12 B written per element), same rotation, same graph trick
    srcs = [torch.empty(3 * T * C, device=dev) for _ in range(sets)]
    dsts = [torch.empty(3 * T * C, device=dev) for _ in range(sets)]
    cgraph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(cgraph):
        for a_, b_ in zip(dsts, srcs):
            a_.copy_(b_)
    cgraph.replay()
    torch.cuda.synchronize()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(reps):
        cgraph.replay()
    c1.record()
    torch.cuda.synchronize()
    copy_us = 1e3 * c0.elapsed_time(c1) / (sets * reps)
    us = 1e3 * e0.elapsed_time(e1) / (sets * reps)
    nbytes = 24.0 * T * C
    hbm = peaks.get("hbm_gbs_sustained") or peaks.get("hbm_gbs")
    ach = nbytes / (us * 1e-6) / 1e9
    return {"kernel": f"hb_gae_returns[T{T},C{C}]", "avg_us": us, "bytes_per_launch": nbytes, "bound": "hbm", "achieved": ach,
            "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
            "same_bytes_copy_us": copy_us, "frac_of_same_size_copy": copy_us / us,
            "how": f"{sets} rotating buffer sets (> L2) x {reps} replays of a CUDA graph of the launches; same_bytes_copy_us = "
                   "torch copy_ kernels moving the same 24 B per element at this size, timed the same way (what a 19.7 MB "
                   "launch can reach at all: launch + fill latency are not amortised at n_rollout_threads=4096)"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        d["_source"] = "MEASURED_PEAKS.json (of measured)"
        return d
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "B200_PROFILING.md fallback (of fallback)"}


REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def _ref_spec(wl, n, steps, warmup, cuda, threads, budget_s):
    """JSON spec for baseline/ref_runner.py: the reference's own argument dicts for this workload."""
    from harl_b200.envs.synthetic import resolve_shapes

    args, algo_args, env_args = make_args(wl, 1, n_override=n)
    shapes = resolve_shapes(args["env"], env_args)
    env_args = {k: v for k, v in env_args.items() if k != "host"}
    env_args["state_type"] = shapes["state_type"]
    if args["env"] in ("smac", "smacv2"):
        # labels only (the env itself is the synthetic one): the SMAC loggers of the reference use np.int (removed from
        # NumPy >= 1.24, SURVEY.md section 8(c)); the MPE logger is the plain base logger
        args = dict(args, env="pettingzoo_mpe")
        env_args.update(scenario="simple_spread_v2", continuous_actions=False)
    spec = dict(args=args, algo_args=algo_args, env_args=env_args, shapes=shapes, n_rollout_threads=n, steps=steps,
                warmup=warmup, cuda=bool(cuda), torch_threads=threads, budget_s=budget_s)
    if env_args.pop("backend", None) == "native":   # the learnable task: the reference runs on the NumPy twin of the CUDA env
        spec["env_kind"] = "mpe_spread"
    return spec


def _ref_subprocess(spec, timeout_s):
    env = {k: v for k, v in os.environ.items() if k not in ("PYTHONPATH", "RANK", "WORLD_SIZE", "LOCAL_RANK")}
    r = subprocess.run([sys.executable, os.path.join(ROOT, "baseline", "ref_runner.py"), json.dumps(spec)],
                       cwd=os.path.join(ROOT, "baseline"), env=env, capture_output=True, text=True, timeout=timeout_s)
    if r.returncode != 0:
        raise RuntimeError("baseline/ref_runner.py failed:\n" + r.stderr[-2000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def reference_run(wl, steps, warmup, n, cuda=False, budget_s=150.0):
    """The UNMODIFIED reference (baseline/_ref, kind "reference") through its own OnPolicy*Runner.run() on this box's
    host cores (or, cuda=True, with device.cuda=True -- the secondary bar of BASELINE.md) at n rollout threads.
    Falls back to the oracle CPU port (kind "port") when baseline/_ref is absent."""
    ncpu = os.cpu_count() or 1
    w = WORKLOADS[wl]
    if not os.path.isdir(os.path.join(REF_DIR, "harl")):
        res = cpu_port_run(wl, max(1, min(steps, 3)), min(warmup, 1), min(n, 512))
        res["fallback"] = "baseline/_ref not present: oracle port"
        return res
    # torch thread count: the reference default (device.torch_threads=4, happo.yaml) and wider settings are probed on a
    # small sample (256 rollout threads, 1 + 1 iterations each); the fastest runs the measurement
    probe = {}
    cands = [4] if cuda else sorted({4, min(16, ncpu), min(32, ncpu)})
    if len(cands) > 1:
        for th in cands:
            probe[th] = _ref_subprocess(_ref_spec(wl, min(n, 256), 1, 1, False, th, 1e9), 600)["seconds_per_step"]
        threads = min(probe, key=probe.get)
    else:
        threads = cands[0]
    out = _ref_subprocess(_ref_spec(wl, n, steps, warmup, cuda, threads, budget_s), 3600)
    dev = "device.cuda=True on cuda:0" if cuda else f"host cores, torch threads={threads} (fastest of {sorted(probe) or cands} on a 256-thread probe)"
    return dict(value=out["value"], unit="env-steps/s", cores=threads, kind="reference", seconds_per_step=out["seconds_per_step"],
                host_cpus=ncpu, thread_probe_s={str(k): round(v, 3) for k, v in probe.items()},
                timed_iterations=out["timed_iterations"], warmup_iterations=out["warmup_iterations"],
                iterations_s=out["iterations_s"], n_rollout_threads=n, cuda=bool(cuda), harl_file=out["harl_file"],
                versions={"torch": out["torch"], "numpy": out["numpy"]},
                sample=f"{w['desc']}" + ("" if n == w["n"] else f" with n_rollout_threads reduced to {n} (the reference is FASTER per env-step on such a sample than at "
                                                            f"the full size -- 46-52 k vs 22-23 k env-steps/s at C2, its rollout buffers no longer fit the "
                                                            f"CPU caches at 4096 threads -- so this in-bench figure flatters it; `--impl reference` runs the full size)") +
                       f"; {out['timed_iterations']} timed iteration(s) after {out['warmup_iterations']} warm-up of the unmodified "
                       f"reference runner (baseline/_ref: pip install --no-deps --target of /root/reference), {dev}")


def cpu_port_run(wl, steps, warmup, n_sample):
    """The CPU oracle port on a bounded sample (n_sample rollout threads) of the workload (cross-check of the reference arm)."""
    import torch

    from harl_b200.envs.synthetic import resolve_shapes
    from oracle.runner import NumpySyntheticEnv, OracleRunner

    args, algo_args, env_args = make_args(wl, 1, n_override=n_sample)
    cfg = {**algo_args["model"], **algo_args["algo"], **algo_args["train"], "algo_name": args["algo"]}
    shapes = resolve_shapes(args["env"], env_args)
    env = NumpySyntheticEnv(shapes, n_sample, seed=1)
    r = OracleRunner(cfg, env, state_type=shapes["state_type"], seed=1)
    r.warmup()
    ncpu = os.cpu_count() or 1
    probe = {}
    for th in sorted({4, min(16, ncpu), min(32, ncpu)}):
        torch.set_num_threads(th)
        t0 = time.perf_counter()
        r.run_iteration()
        probe[th] = time.perf_counter() - t0
    cores = min(probe, key=probe.get)
    torch.set_num_threads(cores)
    for _ in range(max(0, warmup - 1)):
        r.run_iteration()
    t0 = time.perf_counter()
    for _ in range(steps):
        r.run_iteration()
    dt = (time.perf_counter() - t0) / steps
    T = cfg["episode_length"]
    return dict(value=T * n_sample / dt, unit="env-steps/s", cores=cores, kind="port", seconds_per_step=dt,
                host_cpus=ncpu, thread_probe_s={str(k): round(v, 3) for k, v in probe.items()},
                sample=f"{WORKLOADS[wl]['desc']} with n_rollout_threads reduced to {n_sample} "
                       f"(cost is linear in n_rollout_threads); {steps} full iteration(s) of the oracle CPU port, "
                       f"torch threads={cores} (fastest of {sorted(probe)})")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-sample", type=int, default=256, help="n_rollout_threads of the bounded CPU sample")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every GPU keeps the workload's n_rollout_threads; strong: they are divided over the GPUs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-n", type=int, default=0, help="--impl reference: n_rollout_threads (default: the workload's own)")
    ap.add_argument("--ref-cuda", action="store_true", help="--impl reference: device.cuda=True (the reference on the B200)")
    ap.add_argument("--ref-budget-s", type=float, default=150.0, help="--impl reference: wall-time budget of the timed run")
    ap.add_argument("--ref-cross-check", action="store_true", help="--impl reference: also time the oracle CPU port")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--profile-out", default="", help="write the per-kernel event profile of one iteration here")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed iteration computed to DIR/<name>.npy (rank 0)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    # the contract is ONE JSON line on stdout: everything the runner / env print (the reference prints its spaces
    # and progress lines) goes to stderr
    # -- at the file-descriptor level, so that C libraries (NCCL prints its version banner to fd 1) are covered too
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    global STRONG
    STRONG = a.scaling == "strong"
    wl = WORKLOADS[a.workload]
    T = wl["T"]
    base = dict(metric="env-steps/sec (whole box) HAPPO update loop", unit="env-steps/s", n_gpus=a.gpus, steps=a.steps,
                warmup=a.warmup, higher_is_better=True, scaling=a.scaling, vs_baseline=None, dtype="f32", data="synthetic",
                config={"workload": f"{a.workload}: {wl['desc']}",
                        "n_rollout_threads_per_gpu": wl["n"] // (world if a.scaling == "strong" else 1),
                        "episode_length": T, "algo": wl.get("algo_name", "happo"),
                        "l2_policy": "rollout buffers + activations per iteration exceed the 126 MB L2 (no flush needed)"})

    if a.impl == "reference":
        if rank != 0:
            return
        # the unmodified reference at the bench configuration itself (same n_rollout_threads, T, networks), a bounded
        # number of iterations: >= 3 timed ones, stopping once --ref-budget-s of wall time is spent
        n_ref = a.ref_n or wl["n"]
        res = reference_run(a.workload, max(3, a.steps), max(1, min(a.warmup, 1)), n_ref, cuda=a.ref_cuda, budget_s=a.ref_budget_s)
        line = dict(base, impl="reference", value=res["value"], ms_per_step=1e3 * res["seconds_per_step"],
                    cpu_baseline=res, gpu_launches=0,
                    e2e={"value": res["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
        n_glob = wl["n"] * (1 if a.scaling == "strong" else world)
        line["reference"] = {"kind": res["kind"], "n_rollout_threads": n_ref, "same_config": n_ref == n_glob,
                             "global_n_rollout_threads_of_our_arm": n_glob,
                             "timed_iterations": res.get("timed_iterations"), "cuda": bool(a.ref_cuda),
                             "note": "unmodified PKU-MARL/HARL OnPolicy*Runner.run() from baseline/_ref (two shims: tensorboardX "
                                     "stub, synthetic batched env), see baseline/ref_runner.py"}
        if a.ref_cross_check and res["kind"] == "reference":
            line["reference"]["oracle_port_cross_check"] = cpu_port_run(a.workload, 1, 1, min(256, wl["n"]))
        print(json.dumps(line), file=real_stdout, flush=True)
        return

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: harl_b200 has no CPU fallback")
    dist_on = world > 1
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if dist_on:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
    from harl_b200.runners import RUNNER_REGISTRY

    args, algo_args, env_args = make_args(a.workload, world)
    runner = RUNNER_REGISTRY[args["algo"]](args, algo_args, env_args)
    runner.warmup()
    runner.logger.init(10**9)
    sp = runner.envs.action_space[0]
    NET_SHAPES.update(out=(sp.n if sp.__class__.__name__ == "Discrete" else sp.shape[0]), discrete=sp.__class__.__name__ == "Discrete",
                      avail=runner.actor_buffer[0].available_actions is not None)
    ms, launches, clocks = timed_iterations(runner, a.steps, a.warmup, torch, dist_on, sample_clocks=(rank == 0))
    if a.dump_outputs and rank == 0:
        dump_outputs(runner, a.dump_outputs, torch)
    n_global = wl["n"] * (1 if STRONG else world)
    value = T * n_global * a.steps / (ms / 1e3)
    line = dict(base, value=value, ms_per_step=ms / a.steps, gpu_launches=int(launches), clocks=clocks)
    # ---- roofline of the dominant kernel (separate profiled iteration, same stream)
    rows = kernel_profile(runner, torch)
    if rank == 0 and rows:
        line["roofline"] = roofline_of(rows, load_peaks())
        # the two kernels BASELINE.json's north_star names: the GAE scan and the PPO-update (clip-loss) kernel
        named = {"gae": gae_microbench(torch, T, runner.critic_buffer.value_preds[0].numel(), load_peaks()),
                 # the same kernel where launch + fill latency and the T-step serial recurrence are amortised
                 "gae_16x_columns": gae_microbench(torch, T, 16 * runner.critic_buffer.value_preds[0].numel(), load_peaks(), sets=2, reps=3),
                 # opt-in variant (hb_set_gae_impl(2) / HB_GAE_IMPL=2): the carry between time segments by a parallel affine scan
                 "gae_parallel_scan_opt_in": gae_microbench(torch, T, runner.critic_buffer.value_preds[0].numel(), load_peaks(), impl=2),
                 "gae_parallel_scan_opt_in_16x_columns": gae_microbench(torch, T, 16 * runner.critic_buffer.value_preds[0].numel(),
                                                                        load_peaks(), sets=2, reps=3, impl=2)}
        ppo = [r for r in rows if r[0].startswith("fused_actor_update")] or [r for r in rows if r[0].startswith("policy_head_grad")]
        if ppo:
            named["ppo_update"] = dict(kernel=ppo[0][0], launches=ppo[0][1], avg_us=1e3 * ppo[0][2] / ppo[0][1], **_rate(ppo[0], load_peaks()))
        line["roofline"]["named_kernels"] = named
        line["config"]["phases_ms"] = {k: round(v, 3) for k, v in getattr(runner, "phase_ms", {}).items()}
        if dist_on:
            from harl_b200 import dist as _d

            line["config"]["exchanges"] = dict(_d.stats, transport="hb_allreduce_bucket (one-shot, NVLink peer memory)" if _d.stats["p2p"]
                                               else "torch.distributed.all_reduce (NCCL)", note="issued by rank 0 over the whole run")
        if a.profile_out:
            tot = sum(r[2] for r in rows)
            with open(a.profile_out, "w") as fh:
                fh.write(f"# per-kernel CUDA-event profile of the update phase of one {a.workload} iteration (event after every launch)\n")
                fh.write(f"# total {tot:.3f} ms over {sum(r[1] for r in rows)} launches\n")
                for lab, cnt, ms_ in rows:
                    fh.write(f"{lab:48s} n={cnt:6d} total={ms_:9.3f} ms avg={1e3 * ms_ / cnt:8.2f} us share={ms_ / tot:6.3f}\n")
                fh.write("# phases (ms, one iteration): " + json.dumps(getattr(runner, "phase_ms", {})) + "\n")
    env_ms = None
    runner.close()
    del runner
    torch.cuda.empty_cache()
    # ---- end to end: host-resident env (pinned H2D of env outputs, D2H of actions, every rollout step)
    if not a.no_e2e:
        args, algo_args, env_args = make_args(a.workload, world, host_env=True)
        r2 = RUNNER_REGISTRY[args["algo"]](args, algo_args, env_args)
        r2.warmup()
        r2.logger.init(10**9)
        ms2, _, _ = timed_iterations(r2, max(1, min(a.steps, 3)), 1, torch, dist_on)
        k2 = max(1, min(a.steps, 3))
        A, N = r2.num_agents, r2.n_local
        od = r2.envs.observation_space[0].shape[0]
        sd = r2.envs.share_observation_space[0].shape[0]
        aw = r2.actor[0].actor.act_width
        na = r2.actor[0].actor.out_dim if r2.actor_buffer[0].available_actions is not None else 0
        h2d = T * N * (A * od * 4 + sd * 4 + 4 + A + A + A * na * 4)  # obs, state, reward, dones, bad flags, avail
        d2h = T * N * A * aw * 4 + (4 * A + 2) * 8
        if getattr(r2.envs, "h2d_bytes", 0):  # the staged host env counts what it actually copies
            h2d = r2.envs.h2d_bytes // (k2 + 1)
            d2h = r2.envs.d2h_bytes // (k2 + 1) + (4 * A + 2) * 8
        line["e2e"] = {"value": T * n_global * k2 / (ms2 / 1e3), "unit": "env-steps/s", "h2d_bytes_per_step": int(h2d),
                       "d2h_bytes_per_step": int(d2h), "ms_per_step": ms2 / k2,
                       "what": "runner.run_iteration with the env on the host: pinned H2D of obs/state/reward/done/avail and "
                               "D2H of the actions every rollout step, D2H of the train infos every iteration"}
        r2.close()
    # ---- CPU baseline on this box's host cores (rank 0, N=1 only)
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        line["cpu_baseline"] = reference_run(a.workload, 3, 1, min(a.cpu_sample, wl["n"]), budget_s=30.0)
    if rank == 0:
        print(json.dumps(line), file=real_stdout, flush=True)
    if dist_on:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
