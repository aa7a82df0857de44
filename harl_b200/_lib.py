"""ctypes binding of include/harl_b200.h (the only way the host code reaches the kernels).

There is no CPU fallback: if the shared library is missing this module raises at import
time, and every non-zero status from the library raises (HB_ERR_UNSUPPORTED ->
NotImplementedError, everything else -> RuntimeError with hb_last_error()).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_C", "libharl_b200.so")

HB_MAX_LAYERS = 4
HB_MAX_AGENTS = 32
HB_MAX_TENSORS = 40

ACTIVATIONS = {"relu": 0, "tanh": 1, "sigmoid": 2, "leaky_relu": 3, "selu": 4, "hardswish": 5, "identity": 6}
HEAD_DISCRETE, HEAD_BOX, HEAD_VALUE = 0, 1, 2


class NetDesc(C.Structure):
    _fields_ = [
        ("in_dim", C.c_int32), ("n_layers", C.c_int32), ("hidden", C.c_int32 * HB_MAX_LAYERS),
        ("feature_norm", C.c_int32), ("activation", C.c_int32), ("rnn_layers", C.c_int32),
        ("head", C.c_int32), ("out_dim", C.c_int32), ("std_x_coef", C.c_float), ("std_y_coef", C.c_float),
    ]


class NetLayout(C.Structure):
    _fields_ = [
        ("n_tensors", C.c_int32), ("total", C.c_int32),
        ("offset", C.c_int32 * HB_MAX_TENSORS), ("rows", C.c_int32 * HB_MAX_TENSORS),
        ("cols", C.c_int32 * HB_MAX_TENSORS), ("names", (C.c_char * 48) * HB_MAX_TENSORS),
        ("prepared_total", C.c_int32),
    ]


class InsertArgs(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int32), ("n_agents", C.c_int32), ("state_type_fp", C.c_int32),
        ("actor_rnn_row", C.c_int32), ("critic_rnn_row", C.c_int32),
        ("dones", C.c_void_p), ("bad_transition", C.c_void_p),
        ("actor_masks_next", C.c_void_p * HB_MAX_AGENTS), ("actor_active_next", C.c_void_p * HB_MAX_AGENTS),
        ("actor_rnn_next", C.c_void_p * HB_MAX_AGENTS),
        ("critic_masks_next", C.c_void_p), ("critic_bad_next", C.c_void_p), ("critic_rnn_next", C.c_void_p),
        ("rewards", C.c_void_p), ("reward_stride_n", C.c_int64), ("reward_stride_a", C.c_int64),
        ("ep_return", C.c_void_p), ("done_sum", C.c_void_p),
    ]


class CollectArgs(C.Structure):
    _fields_ = [
        ("n_agents", C.c_int32), ("deterministic", C.c_int32), ("rows", C.c_int64), ("offset", C.c_uint64),
        ("actor_desc", C.POINTER(NetDesc) * HB_MAX_AGENTS), ("actor_prepared", C.c_void_p * HB_MAX_AGENTS),
        ("obs", C.c_void_p * HB_MAX_AGENTS), ("avail", C.c_void_p * HB_MAX_AGENTS),
        ("actions", C.c_void_p * HB_MAX_AGENTS), ("logp", C.c_void_p * HB_MAX_AGENTS),
        ("seed", C.c_uint64 * HB_MAX_AGENTS),
        ("critic_desc", C.POINTER(NetDesc)), ("critic_prepared", C.c_void_p), ("share_obs", C.c_void_p),
        ("critic_rows", C.c_int64), ("values", C.c_void_p), ("offset_base", C.c_void_p),
        ("actor_rnn", C.c_void_p * HB_MAX_AGENTS), ("actor_rnn_out", C.c_void_p * HB_MAX_AGENTS),
        ("actor_masks", C.c_void_p * HB_MAX_AGENTS),
        ("critic_rnn", C.c_void_p), ("critic_rnn_out", C.c_void_p), ("critic_masks", C.c_void_p),
    ]


class PPOHyper(C.Structure):
    _fields_ = [("clip_param", C.c_float), ("entropy_coef", C.c_float), ("use_policy_active_masks", C.c_int32),
                ("action_aggregation_prod", C.c_int32), ("use_clip", C.c_int32)]


class ActorBatch(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("actions", C.c_void_p), ("old_logp", C.c_void_p), ("adv", C.c_void_p),
                ("factor", C.c_void_p), ("active", C.c_void_p), ("avail", C.c_void_p), ("index", C.c_void_p),
                ("rows", C.c_int64), ("rnn_states", C.c_void_p), ("masks", C.c_void_p), ("seq_len", C.c_int64)]


class ValueHyper(C.Structure):
    _fields_ = [("clip_param", C.c_float), ("huber_delta", C.c_float), ("value_loss_coef", C.c_float),
                ("use_huber_loss", C.c_int32), ("use_clipped_value_loss", C.c_int32)]


class CriticBatch(C.Structure):
    _fields_ = [("share_obs", C.c_void_p), ("value_preds", C.c_void_p), ("returns", C.c_void_p),
                ("index", C.c_void_p), ("rows", C.c_int64), ("rnn_states", C.c_void_p), ("masks", C.c_void_p),
                ("seq_len", C.c_int64)]


class AdamHyper(C.Structure):
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("weight_decay", C.c_float), ("max_grad_norm", C.c_float), ("use_max_grad_norm", C.c_int32),
                ("step", C.c_int32)]


HB_MPE_MAX_AGENTS = 8


class CopySeg(C.Structure):
    _fields_ = [("dst", C.c_void_p), ("src", C.c_void_p), ("bytes", C.c_int64)]


def copy_segments(dsts, srcs, src_pinned=False, dst_pinned=False):
    """dst[i].copy_(src[i]) for all i in ONE launch (hb_copy_segments).  Either side may be on the device or in PINNED host
    memory (device-accessible under unified addressing: the kernel then reads / writes it over PCIe), not both on the host.  Tensors must
    be contiguous, equal-sized and -typed, hold whole 4-byte words and start on 16-byte boundaries -- returns False (nothing
    done) otherwise, for the caller's fallback.  ``src_pinned``: the caller vouches that host sources are pinned (skips one
    cudaPointerGetAttributes per tensor)."""
    n = len(dsts)
    if n == 0 or n > 16:
        return False
    segs = (CopySeg * n)()
    for i, (d, s) in enumerate(zip(dsts, srcs)):
        nbytes = d.numel() * d.element_size()
        if not ((d.is_cuda or dst_pinned or d.is_pinned()) and (s.is_cuda or src_pinned or s.is_pinned()) and (d.is_cuda or s.is_cuda)
                and d.is_contiguous() and s.is_contiguous() and d.dtype == s.dtype
                and d.numel() == s.numel() and nbytes % 4 == 0 and d.data_ptr() % 16 == 0 and s.data_ptr() % 16 == 0):
            return False
        segs[i].dst, segs[i].src, segs[i].bytes = d.data_ptr(), s.data_ptr(), nbytes
    call("hb_copy_segments", segs, n, stream_ptr())
    return True


class MpeArgs(C.Structure):
    _fields_ = [("n_envs", C.c_int32), ("n_agents", C.c_int32), ("n_landmarks", C.c_int32), ("continuous", C.c_int32),
                ("max_cycles", C.c_int32), ("reset_all", C.c_int32), ("seed", C.c_uint64),
                ("pos", C.c_void_p), ("vel", C.c_void_p), ("landmarks", C.c_void_p), ("step_count", C.c_void_p),
                ("episode", C.c_void_p), ("actions", C.c_void_p * HB_MPE_MAX_AGENTS),
                ("obs_out", C.c_void_p * HB_MPE_MAX_AGENTS), ("share_obs_out", C.c_void_p), ("rewards_out", C.c_void_p),
                ("rewards_na_out", C.c_void_p), ("dones_out", C.c_void_p), ("bad_out", C.c_void_p)]


P = C.c_void_p
# name -> (restype, argtypes); every symbol include/harl_b200.h declares
SIGNATURES = {
    "hb_version": (C.c_int, []),
    "hb_last_error": (C.c_char_p, []),
    "hb_sync_check": (C.c_int, []),
    "hb_kernel_launch_count": (C.c_uint64, []),
    "hb_profile_begin": (C.c_int, [P]),
    "hb_profile_end": (C.c_int, [C.c_char_p, C.c_int]),
    "hb_set_gemm_impl": (C.c_int, [C.c_int]),
    "hb_get_gemm_impl": (C.c_int, []),
    "hb_set_fused_update": (C.c_int, [C.c_int]),
    "hb_get_fused_update": (C.c_int, []),
    "hb_fused_timing_enable": (C.c_int, [C.c_int]),
    "hb_fused_timing_read": (C.c_int, [P]),
    "hb_net_layout_of": (C.c_int, [C.POINTER(NetDesc), C.POINTER(NetLayout)]),
    "hb_net_prepare": (C.c_int, [C.POINTER(NetDesc), P, P, P]),
    "hb_workspace_bytes": (C.c_size_t, [C.POINTER(NetDesc), C.c_int64, C.c_int]),
    "hb_rollout_insert_masks": (C.c_int, [C.POINTER(InsertArgs), P]),
    "hb_rollout_collect": (C.c_int, [C.POINTER(CollectArgs), P, C.c_size_t, P]),
    "hb_counter_add": (C.c_int, [P, C.c_uint64, P]),
    "hb_policy_act": (C.c_int, [C.POINTER(NetDesc), P, P, C.c_int64, P, C.c_int, C.c_uint64, C.c_uint64, P, P, P,
                                C.c_size_t, P]),
    "hb_value_forward": (C.c_int, [C.POINTER(NetDesc), P, P, C.c_int64, P, P, C.c_size_t, P]),
    "hb_copy_segments": (C.c_int, [P, C.c_int32, P]),
    "hb_comm_create": (C.c_int, [C.c_int32, C.c_int32, C.c_size_t, C.POINTER(C.c_void_p), P]),
    "hb_comm_open_peers": (C.c_int, [P, P]),
    "hb_allreduce_bucket": (C.c_int, [P, P, C.c_int64, C.c_int32, P]),
    "hb_comm_status": (C.c_int, [P]),
    "hb_comm_destroy": (C.c_int, [P]),
    "hb_set_gae_impl": (C.c_int, [C.c_int]),
    "hb_get_gae_impl": (C.c_int, []),
    "hb_gae_returns": (C.c_int, [P, P, P, P, P, P, P, C.c_int32, C.c_int64, C.c_float, C.c_float, C.c_int, C.c_int,
                                 P, P]),
    "hb_masked_moments": (C.c_int, [P, P, C.c_int64, P, P]),
    "hb_normalize_by_moments": (C.c_int, [P, P, C.c_int64, P, P]),
    "hb_valuenorm_update": (C.c_int, [P, P, C.c_double, P]),
    "hb_valuenorm_apply": (C.c_int, [P, P, P, C.c_int64, C.c_int, P]),
    "hb_policy_evaluate": (C.c_int, [C.POINTER(NetDesc), P, C.POINTER(ActorBatch), P, P, P, C.c_int, P, C.c_size_t, P]),
    "hb_ppo_actor_grad": (C.c_int, [C.POINTER(NetDesc), P, P, C.POINTER(ActorBatch), C.POINTER(PPOHyper), P, P, P, P,
                                    C.c_size_t, P]),
    "hb_ppo_actor_grad_logp": (C.c_int, [C.POINTER(NetDesc), P, P, C.POINTER(ActorBatch), C.POINTER(PPOHyper), P, P, P, P, P,
                                         C.c_size_t, P]),
    "hb_value_grad": (C.c_int, [C.POINTER(NetDesc), P, P, C.POINTER(CriticBatch), C.POINTER(ValueHyper), P,
                                C.c_double, P, P, P, C.c_size_t, P]),
    "hb_clip_adam_step": (C.c_int, [C.POINTER(NetDesc), P, P, P, P, P, C.POINTER(AdamHyper), P, P]),
    "hb_policy_act_rnn": (C.c_int, [C.POINTER(NetDesc), P, P, C.c_int64, P, P, P, C.c_int, C.c_uint64, C.c_uint64, P, P, P,
                                    P, P, C.c_size_t, P]),
    "hb_value_forward_rnn": (C.c_int, [C.POINTER(NetDesc), P, P, C.c_int64, P, P, P, P, P, C.c_size_t, P]),
    "hb_set_trpo_jvp_impl": (C.c_int, [C.c_int]),
    "hb_get_trpo_jvp_impl": (C.c_int, []),
    "hb_set_rnn_impl": (C.c_int, [C.c_int]),
    "hb_get_rnn_impl": (C.c_int, []),
    "hb_trpo_workspace_bytes": (C.c_size_t, [C.POINTER(NetDesc), C.c_int64]),
    "hb_trpo_old_dist": (C.c_int, [C.POINTER(NetDesc), P, C.POINTER(ActorBatch), P, P, C.c_size_t, P]),
    "hb_trpo_fvp": (C.c_int, [C.POINTER(NetDesc), P, P, C.POINTER(ActorBatch), P, P, C.c_double, C.c_int, P, P,
                              C.c_size_t, P]),
    "hb_trpo_fvp_finish": (C.c_int, [C.POINTER(NetDesc), P, P, P, C.c_float, P]),
    "hb_trpo_eval": (C.c_int, [C.POINTER(NetDesc), P, C.POINTER(ActorBatch), C.POINTER(PPOHyper), P, P, P, P,
                               C.c_size_t, P]),
    "hb_trpo_cg_init": (C.c_int, [P, P, P, P, P, C.c_int, P]),
    "hb_trpo_cg_step": (C.c_int, [P, P, P, P, P, C.c_int, C.c_float, P]),
    "hb_trpo_full_step": (C.c_int, [P, P, P, C.c_float, P, P, C.c_int, P]),
    "hb_trpo_apply_step": (C.c_int, [P, P, P, C.c_float, C.c_int, P]),
    "hb_vec_scale": (C.c_int, [P, C.c_float, C.c_int, P]),
    "hb_mpe_spread_step": (C.c_int, [C.POINTER(MpeArgs), P]),
}

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -m harl_b200.build` (or __graft_entry__.build()). "
        "harl_b200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)
for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args

HB_ERR_UNSUPPORTED = -2
GEMM_IMPLS = {"fp32": 0, "3xtf32": 1}
if os.environ.get("HB_GEMM_IMPL"):
    lib.hb_set_gemm_impl(GEMM_IMPLS[os.environ["HB_GEMM_IMPL"]])
_NO_CHECK = {"hb_version", "hb_last_error", "hb_workspace_bytes", "hb_trpo_workspace_bytes", "hb_kernel_launch_count", "hb_profile_end", "hb_get_gemm_impl", "hb_get_rnn_impl", "hb_get_trpo_jvp_impl", "hb_get_fused_update", "hb_get_gae_impl", "hb_comm_status"}

# launches of library entry points since import (bench.py's gpu_launches bookkeeping)
call_count = 0


def check(rc, what=""):
    if rc == 0:
        return
    msg = lib.hb_last_error().decode(errors="replace")
    if rc == HB_ERR_UNSUPPORTED:
        raise NotImplementedError(f"harl_b200 {what}: {msg}")
    raise RuntimeError(f"harl_b200 {what} failed ({rc}): {msg}")


def call(name, *args):
    """Invoke a status-returning entry point and raise on failure."""
    global call_count
    call_count += 1
    check(getattr(lib, name)(*args), name)


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (or None)."""
    if t is None:
        return None
    assert t.is_contiguous(), "harl_b200 kernels need contiguous tensors"
    return t.data_ptr()


def stream_ptr():
    import torch

    return torch.cuda.current_stream().cuda_stream
