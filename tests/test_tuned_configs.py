"""CPU: every on-policy tuned config of the reference (tuned_configs/*/*/{happo,hatrpo,haa2c,mappo}/config.json) is
structurally inside the device path: its model section maps to an hb_net_desc the library lays out (host-only call),
its algorithm is registered, and the one documented exception (share_param together with a recurrent policy) does not
occur in any of them.  The configs are stored in tests/golden/reference_tuned_configs.json
(tests/golden/make_reference_configs.py)."""
import ctypes as C
import json
import os

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_tuned_configs.json")
ON_POLICY = ("happo", "hatrpo", "haa2c", "mappo")


def test_on_policy_tuned_configs_are_in_scope():
    from harl_b200 import _lib as L
    from harl_b200.algorithms.actors import ALGO_REGISTRY
    from harl_b200.nets import make_desc
    from harl_b200.runners import RUNNER_REGISTRY

    with open(GOLDEN, encoding="utf-8") as fh:
        configs = json.load(fh)
    seen = 0
    for f, blob in configs.items():
        algo = blob["main_args"]["algo"]
        if algo not in ON_POLICY:
            continue
        seen += 1
        assert algo in ALGO_REGISTRY and algo in RUNNER_REGISTRY, f
        model, alg = blob["algo_args"]["model"], blob["algo_args"]["algo"]
        recurrent = bool(model.get("use_recurrent_policy") or model.get("use_naive_recurrent_policy"))
        assert not (recurrent and alg.get("share_param")), f"{f}: share_param + recurrent policy (fails loudly, DESIGN.md 7)"
        for head, in_dim, out_dim in ((L.HEAD_DISCRETE, 30, 12), (L.HEAD_BOX, 30, 3), (L.HEAD_VALUE, 60, 1)):
            d = make_desc(model, in_dim, head, out_dim)
            lay = L.NetLayout()
            rc = L.lib.hb_net_layout_of(C.byref(d), C.byref(lay))
            assert rc == 0, (f, L.lib.hb_last_error())
            assert lay.total > 0 and lay.prepared_total > 0
            names = [lay.names[i].value.decode() for i in range(lay.n_tensors)]
            assert ("rnn.norm.weight" in names) == recurrent, f
    assert seen >= 80
