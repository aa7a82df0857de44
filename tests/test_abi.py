"""CPU checks of the C-ABI library: it loads, exports every declared symbol, and its host-only
entry points (layout, workspace sizing, argument validation) behave.  No kernels run here."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from tests import util as U

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    from harl_b200 import build

    build.build()
    from harl_b200 import _lib

    return _lib


def declared_functions():
    src = open(os.path.join(ROOT, "include", "harl_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hb_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported_and_bound(L):
    names = declared_functions()
    assert len(names) >= 18
    for n in names:
        assert hasattr(L.lib, n), f"{n} declared in include/harl_b200.h but not exported"
        assert n in L.SIGNATURES, f"{n} has no ctypes signature"
    assert set(L.SIGNATURES) == set(names)
    assert L.lib.hb_version() == 100


@pytest.mark.parametrize("tag,head", [("mlp_disc", "Discrete"), ("mlp_box", "Box"), ("gru_disc", "Discrete"),
                                      ("gru_box", "Box"), ("mlp_disc_tanh", "Discrete")])
def test_layout_matches_reference_state_dict(L, tag, head):
    """Flat layout = reference state_dict keys, order and shapes (checkpoint interchange)."""
    from harl_b200.nets import DeviceNet
    from tests.test_oracle_golden import POLICY_CFG

    over, _ = POLICY_CFG[tag]
    cfg = U.base_args(**over)
    g = U.load(f"policy_{tag}")
    ref_actor = [(k[len("actor/"):], g[k].shape) for k in g if k.startswith("actor/")]
    out_dim = g["avail"].shape[1] if head == "Discrete" else g["actions"].shape[1]
    hid = L.HEAD_DISCRETE if head == "Discrete" else L.HEAD_BOX
    net = DeviceNet(cfg, g["obs"].shape[1], hid, out_dim, "cpu", init=False)
    assert [(k, tuple(s)) for k, (_, s) in net.entries.items()] == [(k, tuple(s)) for k, s in ref_actor]
    ref_critic = [(k[len("critic/"):], g[k].shape) for k in g if k.startswith("critic/")]
    cnet = DeviceNet(cfg, g["cobs"].shape[1], L.HEAD_VALUE, 1, "cpu", init=False)
    assert [(k, tuple(s)) for k, (_, s) in cnet.entries.items()] == [(k, tuple(s)) for k, s in ref_critic]
    # offsets are 16-byte aligned and non-overlapping
    end = 0
    for k, (off, shape) in net.entries.items():
        assert off % 4 == 0 and off >= end
        end = off + int(np.prod(shape))
    assert net.total >= end


def test_param_counts_match_survey(L):
    """SURVEY.md Appendix A parameter counts (C1/C2 discrete actor 20 137, critic 24 301; C5 85 140 / 82 929)."""
    from harl_b200.nets import DeviceNet

    cfg = U.base_args(hidden_sizes=[128, 128])
    count = lambda n: sum(int(np.prod(s)) for _, s in n.entries.values())
    assert count(DeviceNet(cfg, 18, L.HEAD_DISCRETE, 5, "cpu", init=False)) == 20137
    assert count(DeviceNet(cfg, 54, L.HEAD_VALUE, 1, "cpu", init=False)) == 24301
    cfg5 = U.base_args(hidden_sizes=[128, 128, 128])
    assert count(DeviceNet(cfg5, 393, L.HEAD_BOX, 1, "cpu", init=False)) == 85140
    assert count(DeviceNet(cfg5, 376, L.HEAD_VALUE, 1, "cpu", init=False)) == 82929


def test_state_dict_roundtrip_and_reference_init_statistics(L):
    import torch

    from harl_b200.nets import DeviceNet

    cfg = U.base_args(hidden_sizes=[64, 64])
    torch.manual_seed(5)
    net = DeviceNet(cfg, 10, L.HEAD_DISCRETE, 4, "cpu", init=True)
    sd = net.state_dict()
    w = sd["base.mlp.fc.0.weight"]
    # orthogonal_ with gain sqrt(2): columns orthogonal, W^T W = 2 I (mlp.py:17-23)
    np.testing.assert_allclose((w.T @ w).numpy(), 2 * np.eye(10), atol=1e-5)
    hw = sd["act.action_out.linear.weight"]
    np.testing.assert_allclose((hw @ hw.T).numpy(), 0.01 ** 2 * np.eye(4), atol=1e-7)
    assert torch.all(sd["base.mlp.fc.2.weight"] == 1) and torch.all(sd["base.mlp.fc.0.bias"] == 0)


def test_unsupported_configs_fail_loudly(L):
    from harl_b200.nets import DeviceNet

    with pytest.raises(NotImplementedError):
        DeviceNet(U.base_args(hidden_sizes=[30, 30]), 8, L.HEAD_DISCRETE, 4, "cpu", init=False)  # not a multiple of 4
    with pytest.raises(NotImplementedError):
        DeviceNet(U.base_args(hidden_sizes=[512]), 8, L.HEAD_DISCRETE, 4, "cpu", init=False)
    with pytest.raises(NotImplementedError):
        DeviceNet(U.base_args(), 8, L.HEAD_DISCRETE, 64, "cpu", init=False)
    net = DeviceNet(U.base_args(), 8, L.HEAD_DISCRETE, 4, "cpu", init=False)
    with pytest.raises(RuntimeError):
        net.prepare()  # no CUDA device -> loud failure, not a CPU fallback


def test_workspace_sizing_and_argument_checks(L):
    from harl_b200.nets import make_desc

    d = make_desc(U.base_args(hidden_sizes=[128, 128]), 18, L.HEAD_DISCRETE, 5)
    small = L.lib.hb_workspace_bytes(C.byref(d), 1000, 0)
    big = L.lib.hb_workspace_bytes(C.byref(d), 10_000_000, 1)
    assert 0 < small < big
    # chunked: workspace stops growing past the chunk size
    assert big == L.lib.hb_workspace_bytes(C.byref(d), 20_000_000, 1)
    rc = L.lib.hb_gae_returns(None, None, None, None, None, None, None, 10, 10, 0.99, 0.94, 1, 1, None, None)
    assert rc == -1 and b"NULL" in L.lib.hb_last_error()


def test_impl_setters_reject_unknown_values(L):
    """hb_set_gemm_impl takes 0 / 1 and hb_set_gae_impl 1 / 2: any other value is refused and changes nothing."""
    gemm, gae = L.lib.hb_get_gemm_impl(), L.lib.hb_get_gae_impl()
    for setter, bad in (("hb_set_gemm_impl", 2), ("hb_set_gae_impl", 0), ("hb_set_gae_impl", 3)):
        assert getattr(L.lib, setter)(bad) == -1 and b"impl must be" in L.lib.hb_last_error()
        assert (L.lib.hb_get_gemm_impl(), L.lib.hb_get_gae_impl()) == (gemm, gae)
    assert L.lib.hb_set_gae_impl(2) == 0 and L.lib.hb_get_gae_impl() == 2
    assert L.lib.hb_set_gae_impl(gae) == 0 and L.lib.hb_get_gae_impl() == gae


def test_recurrent_and_trust_region_workspace_sizing(L):
    """Host-only sizing calls: recurrent batches are never chunked (a chunk would cut every sequence), so their
    workspace keeps growing with the row count; the trust-region workspace covers the gradient workspace plus the
    tangent buffers (and the GRU tangent buffers for recurrent nets)."""
    from harl_b200.nets import make_desc

    mlp = make_desc(U.base_args(hidden_sizes=[64, 64]), 30, L.HEAD_DISCRETE, 12)
    gru = make_desc(U.base_args(hidden_sizes=[64, 64], use_recurrent_policy=True), 30, L.HEAD_DISCRETE, 12)
    gru2 = make_desc(U.base_args(hidden_sizes=[64, 64], use_recurrent_policy=True, recurrent_n=2), 30, L.HEAD_DISCRETE, 12)
    ws = lambda d, rows, mode: L.lib.hb_workspace_bytes(C.byref(d), rows, mode)
    tws = lambda d, rows: L.lib.hb_trpo_workspace_bytes(C.byref(d), rows)
    for rows in (4096, 100_000):
        assert ws(mlp, rows, 0) < ws(gru, rows, 0) < ws(gru2, rows, 0)
        assert ws(mlp, rows, 1) < ws(gru, rows, 1) < ws(gru2, rows, 1)
        assert ws(mlp, rows, 1) < tws(mlp, rows) and ws(gru, rows, 1) < tws(gru, rows)
        assert tws(gru, rows) - ws(gru, rows, 1) > tws(mlp, rows) - ws(mlp, rows, 1)   # GRU tangent buffers
    assert ws(mlp, 20_000_000, 1) == ws(mlp, 10_000_000, 1)        # feed-forward nets: chunked
    assert ws(gru, 4_000_000, 1) > ws(gru, 2_000_000, 1) * 1.9     # recurrent nets: one chunk, linear in the rows
    # argument checks of the new entry points happen before any CUDA call
    assert L.lib.hb_trpo_cg_init(None, None, None, None, None, 10, None) == -1 and b"bad argument" in L.lib.hb_last_error()
    assert L.lib.hb_trpo_full_step(None, None, None, 0.01, None, None, 10, None) == -1
    assert L.lib.hb_vec_scale(None, 1.0, 10, None) == -1
