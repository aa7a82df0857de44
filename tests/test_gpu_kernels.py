"""GPU parity tests: CUDA kernels (through the C-ABI) vs the oracle and the reference's golden vectors.

Tolerances (fp32 everywhere, reference = PyTorch CPU fp32):
  * masks / GAE returns / advantages: bit-exact
  * log-probs, values, entropies: 2e-5 abs (different summation order inside the GEMMs)
  * gradients: 2e-4 relative to the tensor's max magnitude; updated weights 2e-5 abs
"""
import ctypes as C

import numpy as np
import pytest
import torch

from tests import util as U

pytestmark = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


def _cu(x, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype).to(_dev()).contiguous()


def _net(cfg, in_dim, head, out_dim, params):
    from harl_b200 import _lib as L
    from harl_b200.nets import DeviceNet

    hid = {"Discrete": L.HEAD_DISCRETE, "Box": L.HEAD_BOX, "value": L.HEAD_VALUE}[head]
    net = DeviceNet(cfg, in_dim, hid, out_dim, _dev(), init=False)
    net.load_state_dict(params)
    return net


# ------------------------------------------------------------------ GAE
def _run_gae(rew, vp, masks, bad, nv, gamma, lam, use_gae, ptl, vn_state):
    from harl_b200 import _lib as L

    T = rew.shape[0]
    Cc = int(np.prod(rew.shape[1:]))
    d_rew, d_vp, d_m, d_b, d_nv = (_cu(x.reshape(x.shape[0], -1)) for x in (rew, vp, masks, bad, nv[None]))
    ret = torch.zeros(T + 1, Cc, device=_dev())
    adv = torch.zeros(T, Cc, device=_dev())
    vn = _cu(vn_state) if vn_state is not None else None
    L.call("hb_gae_returns", L.ptr(d_rew), L.ptr(d_vp), L.ptr(d_m), L.ptr(d_b), L.ptr(d_nv), L.ptr(ret), L.ptr(adv), T,
           Cc, float(np.float32(gamma)), float(np.float32(gamma * lam)), int(use_gae), int(ptl), L.ptr(vn),
           L.stream_ptr())
    torch.cuda.synchronize()
    return ret.cpu().numpy(), d_vp.cpu().numpy(), adv.cpu().numpy()


@pytest.mark.parametrize("name", U.names("gae_"))
def test_gae_golden_bit_exact(name):
    g = U.load(name)
    use_gae, ptl, use_vn = (int(name.split(k)[1][0]) for k in ("_gae", "_ptl", "_vn"))
    vn = np.array([g["vn_mean"][0], g["vn_mean_sq"][0], g["vn_debias"]], np.float32) if use_vn else None
    ret, vp, adv = _run_gae(g["in.rewards"], g["in.value_preds"], g["in.masks"], g["in.bad_masks"], g["next_value"],
                            float(g["gamma"]), float(g["gae_lambda"]), use_gae, ptl, vn)
    shp = g["returns"].shape
    assert np.array_equal(ret[:-1].reshape(shp[0] - 1, *shp[1:]), g["returns"][:-1])
    if use_gae:
        assert np.array_equal(vp.reshape(shp), g["value_preds"])
    else:
        assert np.array_equal(ret[-1].reshape(shp[1:]), g["returns"][-1])
    assert np.array_equal(adv.reshape(g["advantages"].shape), g["advantages"])


@pytest.fixture(params=[1], ids=["seg"])
def sequential_carry(request):
    """hb_set_gae_impl(1) for the test, whatever HB_GAE_IMPL selected: the bit-exact assertions hold for the sequential
    carry between time segments, not for the parallel scan."""
    from harl_b200 import _lib as L

    prev = L.lib.hb_get_gae_impl()
    L.call("hb_set_gae_impl", request.param)
    yield request.param
    L.call("hb_set_gae_impl", prev)


# T <= 256 with GAE runs the time-segmented kernel (gae_seg.cu); longer rollouts and the branch without GAE run the
# column tiles of gae.cu (every tile width 32 / 16 / 8 / 4 occurs below), or one thread per column when C % 4 != 0
@pytest.mark.parametrize("C_,T", [(4096, 200), (1024 * 6, 50), (8, 200), (4099, 33), (100, 256), (64, 257), (37, 5), (4096, 129),
                                  (4096, 300), (4099, 300), (8, 1000), (1024 * 6, 257), (100, 512), (37, 999), (2048, 1000),
                                  (256, 2000), (4096, 512), (4097, 257)])
@pytest.mark.parametrize("flags", [(1, 1, 1), (1, 0, 0), (0, 1, 1), (0, 0, 0)])
def test_gae_large_vs_oracle(C_, T, flags, sequential_carry):
    """BASELINE sizes and ragged widths / lengths vs the oracle, bit-exact."""
    from oracle import buffers as ob

    use_gae, ptl, use_vn = flags
    rng = np.random.default_rng(C_ + T)
    rew = rng.standard_normal((T, C_, 1)).astype(np.float32)
    vp = rng.standard_normal((T + 1, C_, 1)).astype(np.float32)
    masks = (rng.random((T + 1, C_, 1)) > 0.05).astype(np.float32)
    bad = np.where((masks == 0) & (rng.random(masks.shape) < 0.5), 0, 1).astype(np.float32)
    nv = rng.standard_normal((C_, 1)).astype(np.float32)
    vn = None
    vs = None
    if use_vn:
        vn = ob.ValueNormState()
        vn.update(rng.standard_normal(500) * 3 + 2)
        vs = np.array([vn.running_mean, vn.running_mean_sq, vn.debiasing_term], np.float32)
    ret_o, vp_o = ob.compute_returns(rew, vp, masks, bad, nv, 0.99, 0.95, bool(use_gae), bool(ptl), vn)
    adv_o = ob.advantages(ret_o, vp_o, vn)
    ret, vpo, adv = _run_gae(rew, vp, masks, bad, nv, 0.99, 0.95, use_gae, ptl, vs)
    assert np.array_equal(ret[:-1].reshape(T, C_, 1), ret_o[:-1])
    assert np.array_equal(adv.reshape(T, C_, 1), adv_o)
    if use_gae:
        assert np.array_equal(vpo.reshape(T + 1, C_, 1), vp_o)
    else:
        assert np.array_equal(ret[-1].reshape(C_, 1), ret_o[-1])


@pytest.mark.parametrize("C_,T,ptl,use_vn", [(4096, 200, 1, 1), (4099, 33, 0, 0), (96, 256, 1, 0), (1000, 7, 0, 1)])
def test_gae_parallel_scan_within_1e6_of_sequential(C_, T, ptl, use_vn):
    """hb_set_gae_impl(2): the carry between time segments comes from a parallel affine scan (FMAs) instead of the
    sequential hand-over.  Stated tolerance: 1e-6 of max|advantage| (the steps inside a segment are replayed exactly)."""
    from harl_b200 import _lib as L

    rng = np.random.default_rng(C_ * 7 + T)
    rew = rng.standard_normal((T, C_, 1)).astype(np.float32)
    vp = rng.standard_normal((T + 1, C_, 1)).astype(np.float32)
    masks = (rng.random((T + 1, C_, 1)) > 0.02).astype(np.float32)
    bad = np.where((masks == 0) & (rng.random(masks.shape) < 0.5), 0, 1).astype(np.float32)
    nv = rng.standard_normal((C_, 1)).astype(np.float32)
    vs = np.array([0.3, 1.9, 0.8], np.float32) if use_vn else None
    out = {}
    for impl in (1, 2):
        L.call("hb_set_gae_impl", impl)
        try:
            out[impl] = _run_gae(rew, vp, masks, bad, nv, 0.99, 0.95, 1, ptl, vs)
        finally:
            L.call("hb_set_gae_impl", 1)
    (ret1, vp1, adv1), (ret2, vp2, adv2) = out[1], out[2]
    assert np.array_equal(vp1, vp2)
    scale = np.abs(adv1).max()
    assert np.abs(adv2 - adv1).max() <= 1e-6 * scale
    assert np.abs(ret2[:-1] - ret1[:-1]).max() <= 1e-6 * max(scale, np.abs(ret1[:-1]).max())
    assert (adv1 == adv2).mean() > 0.5   # most entries are identical: only the carried term differs by an ulp or two


def test_gae_linearity_in_rewards():
    """Size-independent property: without ValueNorm/time limits, returns are linear in (rewards, values)."""
    rng = np.random.default_rng(0)
    T, C_ = 200, 4096
    masks = (rng.random((T + 1, C_, 1)) > 0.05).astype(np.float32)
    bad = np.ones_like(masks)
    z = np.zeros((T + 1, C_, 1), np.float32)
    r1 = rng.standard_normal((T, C_, 1)).astype(np.float32)
    ret1, _, _ = _run_gae(r1, z, masks, bad, z[0], 0.99, 0.95, 1, 0, None)
    ret2, _, _ = _run_gae(2 * r1, z, masks, bad, z[0], 0.99, 0.95, 1, 0, None)
    np.testing.assert_allclose(ret2, 2 * ret1, rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------ insert masks
@pytest.mark.parametrize("st", ["EP", "FP"])
def test_insert_masks_bit_exact(st):
    from harl_b200 import _lib as L

    g = U.load(f"insert_{st}")
    T, N, A = g["dones"].shape
    h = g["a0.rnn_states"].shape[-1]
    for t in range(T):
        a = L.InsertArgs()
        a.n_envs, a.n_agents, a.state_type_fp = N, A, int(st == "FP")
        a.actor_rnn_row, a.critic_rnn_row = h, h
        dones, bad = _cu(g["dones"][t], torch.uint8), _cu(g["bad"][t], torch.uint8)
        a.dones, a.bad_transition = L.ptr(dones), L.ptr(bad)
        am = [torch.full((N,), 7.0, device=_dev()) for _ in range(A)]
        aa = [torch.full((N,), 7.0, device=_dev()) for _ in range(A)]
        ar = [torch.ones(N, h, device=_dev()) for _ in range(A)]
        for i in range(A):
            a.actor_masks_next[i], a.actor_active_next[i], a.actor_rnn_next[i] = L.ptr(am[i]), L.ptr(aa[i]), L.ptr(ar[i])
        cshape = (N,) if st == "EP" else (N, A)
        cm, cb = torch.full(cshape, 7.0, device=_dev()), torch.full(cshape, 7.0, device=_dev())
        cr = torch.ones(*cshape, h, device=_dev())
        a.critic_masks_next, a.critic_bad_next, a.critic_rnn_next = L.ptr(cm), L.ptr(cb), L.ptr(cr)
        L.call("hb_rollout_insert_masks", C.byref(a), L.stream_ptr())
        torch.cuda.synchronize()
        denv = g["dones"][t].all(1)
        for i in range(A):
            assert np.array_equal(am[i].cpu().numpy(), g[f"a{i}.masks"][t + 1][:, 0])
            assert np.array_equal(aa[i].cpu().numpy(), g[f"a{i}.active_masks"][t + 1][:, 0])
            assert np.array_equal(ar[i].cpu().numpy()[:, 0] == 0, denv)
        assert np.array_equal(cm.cpu().numpy().reshape(g["c.masks"][t + 1].shape), g["c.masks"][t + 1])
        assert np.array_equal(cb.cpu().numpy().reshape(g["c.bad_masks"][t + 1].shape), g["c.bad_masks"][t + 1])
        assert np.array_equal((cr.cpu().numpy().reshape(N, -1) == 0).all(1), denv)


# ------------------------------------------------------------------ moments / ValueNorm
def test_masked_moments_and_normalize():
    from harl_b200 import _lib as L
    from oracle import buffers as ob

    rng = np.random.default_rng(3)
    x = (rng.standard_normal((200, 4096, 1)) * 2 + 0.3).astype(np.float32)
    w = (rng.random(x.shape) > 0.3).astype(np.float32)
    dx, dw = _cu(x), _cu(w)
    m3 = torch.zeros(3, dtype=torch.float64, device=_dev())
    L.call("hb_masked_moments", L.ptr(dx), L.ptr(dw), x.size, L.ptr(m3), L.stream_ptr())
    y = torch.empty_like(dx)
    L.call("hb_normalize_by_moments", L.ptr(dx), L.ptr(y), x.size, L.ptr(m3), L.stream_ptr())
    ref, mean, std = ob.normalize_advantages(x, w)
    s, q, c = m3.cpu().numpy()
    assert c == w.sum()
    np.testing.assert_allclose(s / c, mean, rtol=1e-5)
    np.testing.assert_allclose(np.sqrt(q / c - (s / c) ** 2), std, rtol=1e-5)
    np.testing.assert_allclose(y.cpu().numpy(), ref, rtol=1e-5, atol=2e-6)


def test_valuenorm_matches_reference():
    from harl_b200 import _lib as L

    g = U.load("valuenorm")
    vn = torch.zeros(3, device=_dev())
    for x, st in zip(g["xs"], g["states"]):
        dx = _cu(x)
        m3 = torch.zeros(3, dtype=torch.float64, device=_dev())
        L.call("hb_masked_moments", L.ptr(dx), None, x.size, L.ptr(m3), L.stream_ptr())
        L.call("hb_valuenorm_update", L.ptr(vn), L.ptr(m3), 0.99999, L.stream_ptr())
        np.testing.assert_allclose(vn.cpu().numpy(), st, rtol=2e-6, atol=1e-10)
    q = _cu(g["q"])
    out = torch.empty_like(q)
    L.call("hb_valuenorm_apply", L.ptr(vn), L.ptr(q), L.ptr(out), q.numel(), 0, L.stream_ptr())
    np.testing.assert_allclose(out.cpu().numpy(), g["norm"], rtol=1e-5, atol=1e-6)
    L.call("hb_valuenorm_apply", L.ptr(vn), L.ptr(q), L.ptr(out), q.numel(), 1, L.stream_ptr())
    np.testing.assert_allclose(out.cpu().numpy(), g["denorm"], rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------ policy / value forward
POLICY_CFG = {
    "mlp_disc": ({}, "Discrete"),
    "mlp_box": (dict(hidden_sizes=[32, 32, 32]), "Box"),
    "mlp_disc_tanh": (dict(activation_func="tanh", use_feature_normalization=False), "Discrete"),
}


@pytest.mark.parametrize("tag", sorted(POLICY_CFG))
def test_policy_forward_golden(tag):
    from harl_b200.nets import DeviceNet

    over, head = POLICY_CFG[tag]
    cfg = U.base_args(**over)
    g = U.load(f"policy_{tag}")
    od = g["obs"].shape[1]
    out_dim = g["avail"].shape[1] if head == "Discrete" else g["actions"].shape[1]
    net = _net(cfg, od, head, out_dim, U.params_of(g, "actor/"))
    obs, acts = _cu(g["obs"]), _cu(g["actions"])
    avail = _cu(g["avail"]) if "avail" in g else None
    B = obs.shape[0]
    logp = torch.zeros(B, net.act_width, device=_dev())
    net.evaluate(DeviceNet.actor_batch(obs, acts, avail=avail), logp_out=logp)
    np.testing.assert_allclose(logp.cpu().numpy(), g["row.logp"], rtol=1e-5, atol=2e-5)
    a = torch.zeros(B, net.act_width, device=_dev())
    lp = torch.zeros(B, net.act_width, device=_dev())
    net.act(obs, avail, True, 0, 0, a, lp)
    if head == "Discrete":
        assert np.array_equal(a.cpu().numpy(), g["det_action"])
    else:
        np.testing.assert_allclose(a.cpu().numpy(), g["det_action"], rtol=1e-5, atol=2e-5)
    np.testing.assert_allclose(lp.cpu().numpy(), g["det_logp"], rtol=1e-5, atol=2e-5)
    critic = _net(cfg, g["cobs"].shape[1], "value", 1, U.params_of(g, "critic/"))
    v = torch.zeros(B, 1, device=_dev())
    critic.values(_cu(g["cobs"]), v)
    np.testing.assert_allclose(v.cpu().numpy(), g["row.values"], rtol=1e-5, atol=2e-5)


@pytest.mark.parametrize("head,na", [("Discrete", 5), ("Discrete", 12), ("Box", 3)])
def test_sampler_statistics(head, na):
    """RNG parity with torch is impossible by construction: check the sampler against the distribution."""
    from oracle import nets as on

    cfg = U.base_args(hidden_sizes=[64, 64])
    torch.manual_seed(0)
    p = on.init_params(cfg, 10, head, na)
    for k in p:
        if "action_out" in k and k.endswith("weight"):
            p[k] = p[k] * 50  # make the distribution non-uniform
    net = _net(cfg, 10, head, na, p)
    B = 200_000
    obs1 = torch.randn(1, 10)
    obs = obs1.repeat(B, 1).to(_dev()).contiguous()
    a = torch.zeros(B, net.act_width, device=_dev())
    lp = torch.zeros(B, net.act_width, device=_dev())
    avail = None
    if head == "Discrete":
        av = torch.ones(1, na)
        av[0, 0] = 0
        avail = av.repeat(B, 1).to(_dev()).contiguous()
    net.act(obs, avail, False, 1234, 5, a, lp)
    a2 = torch.zeros_like(a)
    net.act(obs, avail, False, 1234, 6, a2, lp.clone())
    assert not torch.equal(a, a2), "different offsets must give different draws"
    feat, _ = on.features(p, cfg, obs1, None, None)
    if head == "Discrete":
        logits = on.categorical_logits(p, feat, av)
        probs = logits.exp()[0].numpy()
        freq = np.bincount(a.cpu().numpy()[:, 0].astype(int), minlength=na) / B
        assert freq[0] == 0.0
        np.testing.assert_allclose(freq, probs, atol=4 * np.sqrt(0.25 / B) + 1e-4)
        np.testing.assert_allclose(lp.cpu().numpy()[:, 0], logits[0].numpy()[a.cpu().numpy()[:, 0].astype(int)], atol=2e-5)
    else:
        mean, std = on.gaussian_params(p, cfg, feat)
        s = a.cpu().numpy()
        np.testing.assert_allclose(s.mean(0), mean[0].numpy(), atol=float(5 * std[0].numpy().max() / np.sqrt(B) + 1e-4))
        np.testing.assert_allclose(s.std(0), std[0].numpy(), rtol=0.02)


# ------------------------------------------------------------------ one HAPPO / critic update
def _tol_grad(got, ref, rel=2e-4):
    scale = max(np.abs(ref).max(), 1e-6)
    np.testing.assert_allclose(got, ref, rtol=0, atol=rel * scale)


@pytest.mark.parametrize("name", U.names("single_update_"))
def test_single_update_golden(name):
    from harl_b200 import _lib as L
    from harl_b200.nets import DeviceNet

    g = U.load(name)
    cfg, m = U.cfg_of(g), U.meta_of(g)
    T, N = cfg["episode_length"], cfg["n_rollout_threads"]
    net = _net(cfg, m["od"], m["head"], m["act_dim"], U.params_of(g, "actor0/"))
    fl = lambda a: _cu(a.reshape(T * N, -1))
    active = fl(g["a0.active_masks"][:-1])
    avail = fl(g["a0.available_actions"][:-1]) if "a0.available_actions" in g else None
    batch = DeviceNet.actor_batch(fl(g["a0.obs"][:-1]), fl(g["a0.actions"]), fl(g["a0.action_log_probs"]),
                                  fl(g["adv"]), fl(g["factor"]), active, avail)
    hyper = L.PPOHyper(cfg["clip_param"], cfg["entropy_coef"], 1, 1, 1)
    norm3 = torch.tensor([0, 0, float(g["a0.active_masks"][:-1].sum())], dtype=torch.float64, device=_dev())
    scal = torch.zeros(4, dtype=torch.float64, device=_dev())
    net.actor_grad(batch, hyper, norm3, scal)
    torch.cuda.synchronize()
    s = scal.cpu().numpy()
    nrm = norm3[2].item()
    ref_pl, ref_ent, ref_gn, ref_ratio = g["actor_scalars"]
    np.testing.assert_allclose([s[0] / nrm, s[1] / nrm, s[2] / s[3]], [ref_pl, ref_ent, ref_ratio], rtol=2e-5, atol=2e-6)
    grads = {k: v.cpu().numpy() for k, v in net.views(net.grad).items()}
    gn = np.sqrt(sum((v.astype(np.float64) ** 2).sum() for v in grads.values()))
    np.testing.assert_allclose(gn, ref_gn, rtol=2e-4)
    coef = min(1.0, cfg["max_grad_norm"] / (ref_gn + 1e-6))
    for k, v in grads.items():
        _tol_grad(v * coef, g["grad.actor0/" + k])
    net.adam_step(cfg["lr"], cfg["opti_eps"], cfg["weight_decay"], cfg["max_grad_norm"], cfg["use_max_grad_norm"])
    np.testing.assert_allclose(net.grad_norm.item(), ref_gn, rtol=2e-4)
    for k, v in net.views().items():
        np.testing.assert_allclose(v.cpu().numpy(), g["out.actor0/" + k], rtol=0, atol=2e-5)

    # ---- critic
    from oracle import buffers as ob
    cnet = _net(cfg, m["sd"], "value", 1, U.params_of(g, "critic/"))
    vn = _cu(g["vn_in"])
    ret = fl(g["c.returns"][:-1])
    m3 = torch.zeros(3, dtype=torch.float64, device=_dev())
    L.call("hb_masked_moments", L.ptr(ret), None, ret.numel(), L.ptr(m3), L.stream_ptr())
    L.call("hb_valuenorm_update", L.ptr(vn), L.ptr(m3), 0.99999, L.stream_ptr())
    cb = DeviceNet.critic_batch(fl(g["c.share_obs"][:-1]), fl(g["c.value_preds"][:-1]), ret, None, T * N)
    vh = L.ValueHyper(cfg["clip_param"], cfg["huber_delta"], cfg["value_loss_coef"], 1, 1)
    cs = torch.zeros(4, dtype=torch.float64, device=_dev())
    cnet.value_grad(cb, vh, vn, 1.0 / (T * N), cs)
    torch.cuda.synchronize()
    c = cs.cpu().numpy()
    ref_vl, ref_cgn = g["critic_scalars"]
    np.testing.assert_allclose(c[0] / c[1], ref_vl, rtol=2e-5)
    cgrads = {k: v.cpu().numpy() for k, v in cnet.views(cnet.grad).items()}
    cgn = np.sqrt(sum((v.astype(np.float64) ** 2).sum() for v in cgrads.values()))
    np.testing.assert_allclose(cgn, ref_cgn, rtol=2e-4)
    coef = min(1.0, cfg["max_grad_norm"] / (ref_cgn + 1e-6))
    for k, v in cgrads.items():
        _tol_grad(v * coef, g["grad.critic/" + k])
    cnet.adam_step(cfg["critic_lr"], cfg["opti_eps"], cfg["weight_decay"], cfg["max_grad_norm"], cfg["use_max_grad_norm"])
    for k, v in cnet.views().items():
        np.testing.assert_allclose(v.cpu().numpy(), g["out.critic/" + k], rtol=0, atol=2e-5)


@pytest.mark.parametrize("shape", [dict(od=18, hs=[128, 128], head="Discrete", na=5, rows=70_000),
                                   dict(od=23, hs=[128, 128, 128], head="Box", na=1, rows=40_000),
                                   dict(od=393, hs=[128, 128, 128], head="Box", na=1, rows=9_000),
                                   dict(od=54, hs=[256, 256], head="Discrete", na=7, rows=5_000),
                                   dict(od=30, hs=[64], head="Discrete", na=12, rows=3_001)])
def test_actor_grad_vs_oracle_baseline_shapes(shape):
    """BASELINE network shapes, multi-chunk row counts, random gather index: grads vs CPU autograd."""
    from harl_b200 import _lib as L
    from harl_b200.nets import DeviceNet
    from oracle import algo as oa
    from oracle import nets as on

    torch.manual_seed(1)
    rng = np.random.default_rng(2)
    cfg = U.base_args(hidden_sizes=shape["hs"], clip_param=0.2, entropy_coef=0.01)
    od, head, na, R = shape["od"], shape["head"], shape["na"], shape["rows"]
    p = on.init_params(cfg, od, head, na)
    for k in p:
        p[k] = p[k] + 0.05 * torch.randn_like(p[k])
    net = _net(cfg, od, head, na, p)
    Rbuf = R + 100
    obs = rng.standard_normal((Rbuf, od)).astype(np.float32)
    ad = 1 if head == "Discrete" else na
    if head == "Discrete":
        avail = (rng.random((Rbuf, na)) < 0.8).astype(np.float32)
        avail[:, 1] = 1
        acts = np.array([[rng.choice(np.flatnonzero(avail[i]))] for i in range(Rbuf)], np.float32)
    else:
        avail, acts = None, rng.standard_normal((Rbuf, ad)).astype(np.float32) * 0.3
    old_lp = (-np.abs(rng.standard_normal((Rbuf, ad))) * 0.3 - 1.0).astype(np.float32)
    adv = rng.standard_normal((Rbuf, 1)).astype(np.float32)
    factor = (1 + 0.2 * rng.standard_normal((Rbuf, 1))).astype(np.float32)
    active = (rng.random((Rbuf, 1)) > 0.15).astype(np.float32)
    index = rng.permutation(Rbuf)[:R].astype(np.int32)
    # oracle, in float64 (the yardstick) and in float32 (the reference's own arithmetic: its distance from the
    # float64 result is the noise floor of these heavily cancelling sums)
    def oracle_grads(dt):
        pg = {k: v.clone().to(dt).requires_grad_(True) for k, v in p.items()}
        t = lambda a: torch.from_numpy(a[index]).to(dt)
        lp_, ent_, _, _ = on.actor_evaluate(pg, cfg, head, t(obs), None, t(acts), None,
                                            t(avail) if avail is not None else None, t(active))
        pl_, total_, imp_ = oa.ppo_loss(lp_, t(old_lp), t(adv), t(active), t(factor), ent_, cfg)
        gs = torch.autograd.grad(total_, list(pg.values()))
        return {k: g.double().numpy() for k, g in zip(pg.keys(), gs)}, pl_, ent_, imp_

    ref, pl, ent, imp = oracle_grads(torch.float64)
    ref32 = oracle_grads(torch.float32)[0]
    # device
    batch = DeviceNet.actor_batch(_cu(obs), _cu(acts), _cu(old_lp), _cu(adv), _cu(factor), _cu(active),
                                  _cu(avail) if avail is not None else None, _cu(index, torch.int32))
    hyper = L.PPOHyper(cfg["clip_param"], cfg["entropy_coef"], 1, 1, 1)
    norm3 = torch.tensor([0, 0, float(active[index].sum())], dtype=torch.float64, device=_dev())
    scal = torch.zeros(4, dtype=torch.float64, device=_dev())
    net.actor_grad(batch, hyper, norm3, scal)
    torch.cuda.synchronize()
    s = scal.cpu().numpy()
    np.testing.assert_allclose([s[0] / norm3[2].item(), s[1] / norm3[2].item(), s[2] / s[3]],
                               [pl.item(), ent.item(), imp.mean().item()], rtol=5e-5, atol=5e-6)
    for k, v in net.views(net.grad).items():
        # Every entry is a sum over up to 70k rows whose terms cancel down to the random-walk magnitude, so errors are
        # stated against the tensor max.  The reference's own fp32 autograd sits 3e-5 .. 1e-4 of the max away from the
        # float64 result; the device (per-row FMA / intrinsic differences, sequential row order) is allowed 2e-3 at the
        # worst entry (3e-3 for the feature-norm affine grads, which cancel hardest) and 3e-4 on average.
        got, want = v.cpu().numpy().astype(np.float64), ref[k]
        scale = max(np.abs(want).max(), 1e-6)
        err = np.abs(got - want)
        floor = np.abs(ref32[k] - want).max()
        lim = (3e-3 if "feature_norm" in k else 2e-3) * scale
        assert err.max() <= max(lim, 16 * floor), (k, err.max() / scale, floor / scale)
        assert err.mean() <= 3e-4 * scale, (k, err.mean() / scale)
    # log-prob sweep on the same rows + factor update (identity batch)
    lp_dev = torch.zeros(Rbuf, ad, device=_dev())
    fac = _cu(factor.copy())
    b2 = DeviceNet.actor_batch(_cu(obs), _cu(acts), avail=_cu(avail) if avail is not None else None)
    net.evaluate(b2, logp_out=lp_dev, logp_ref=_cu(old_lp), factor_inout=fac, agg_prod=True)
    with torch.no_grad():
        lp_all, _, _, _ = on.actor_evaluate(p, cfg, head, torch.from_numpy(obs), None, torch.from_numpy(acts), None,
                                            torch.from_numpy(avail) if avail is not None else None, None)
    np.testing.assert_allclose(lp_dev.cpu().numpy(), lp_all.numpy(), rtol=1e-5, atol=3e-5)
    ref_fac = oa.factor_update(factor, lp_all, torch.from_numpy(old_lp), cfg)
    np.testing.assert_allclose(fac.cpu().numpy().reshape(-1, 1), ref_fac, rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("act", ["hardswish", "identity"])
def test_activations_the_reference_cannot_build_raise_the_same_error(act):
    """models_tools.py:28-50 lists hardswish and identity, but every MLP goes through mlp.py:20
    nn.init.calculate_gain(activation_func), which rejects both: the reference raises ValueError at construction
    (tests/golden/make_golden.py `activations` records it), and so does DeviceNet."""
    from harl_b200 import _lib as L
    from harl_b200.nets import DeviceNet

    with pytest.raises(ValueError, match="Unsupported nonlinearity"):
        DeviceNet(U.base_args(activation_func=act), 12, L.HEAD_DISCRETE, 5, "cuda:0")


def test_copy_segments_equals_elementwise_copies():
    """hb_copy_segments: every segment copied exactly, tails shorter than 16 bytes included, neighbours untouched."""
    from harl_b200 import _lib as L

    g = torch.Generator().manual_seed(5)
    sizes = [4096 * 18, 4096 * 54, 4096, 7, 4, 1, 4096 * 5 + 3, 16]
    srcs = [torch.randn(n + 8, generator=g).to(_dev())[4:4 + n] for n in sizes]          # 16-byte aligned interior views
    dsts = [torch.full((n + 8,), -7.0, device=_dev())[4:4 + n] for n in sizes]
    assert L.copy_segments(dsts, srcs)
    torch.cuda.synchronize()
    for d, s in zip(dsts, srcs):
        assert torch.equal(d, s)
        full = d._base if d._base is not None else d
        assert (full[:4] == -7.0).all() and (full[-4:] == -7.0).all()
    # sources in pinned host memory: the kernel reads them over PCIe (the host env's step outputs take this path)
    hsrc = [torch.randn(n, generator=g).pin_memory() for n in (4096 * 18, 12, 4096)] + [torch.randint(0, 2, (4096, 3), dtype=torch.uint8).pin_memory()]
    hdst = [torch.zeros(t.shape, dtype=t.dtype, device=_dev()) for t in hsrc]
    assert L.copy_segments(hdst, hsrc)
    torch.cuda.synchronize()
    for d, s in zip(hdst, hsrc):
        assert torch.equal(d.cpu(), s)
    back = [torch.zeros(t.shape, dtype=t.dtype).pin_memory() for t in hsrc]             # device -> pinned host (the actions' way)
    assert L.copy_segments(back, hdst)
    torch.cuda.synchronize()
    for b, s in zip(back, hsrc):
        assert torch.equal(b, s)
    assert not L.copy_segments([torch.zeros(8, device=_dev())], [torch.zeros(8)])   # pageable host memory: declined
    assert not L.copy_segments([torch.zeros(8).pin_memory()], [torch.zeros(8).pin_memory()])   # host -> host: not this kernel's job
    ints = [torch.arange(100, dtype=torch.int32, device=_dev())]
    outs = [torch.zeros(100, dtype=torch.int32, device=_dev())]
    assert L.copy_segments(outs, ints) and torch.equal(outs[0], ints[0])
    assert not L.copy_segments([torch.zeros(9, device=_dev())[1:]], [torch.zeros(9, device=_dev())[1:]])   # misaligned: declined
    assert not L.copy_segments([torch.zeros(4, 4, device=_dev()).t()], [torch.zeros(4, 4, device=_dev())])   # not contiguous
