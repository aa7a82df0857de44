"""The reference's examples/train.py (PKU-MARL/HARL) drives this package through the `harl` alias: it imports
harl.utils.configs_tools and harl.runners.RUNNER_REGISTRY, builds the configuration from this repo's yaml defaults / a
tuned config.json, applies the command-line overrides and constructs RUNNER_REGISTRY[algo](args, algo_args, env_args)
-> run() -> close().  What the unmodified reference train.py handed to the runner for the command lines below is stored
in tests/golden/reference_train_py.json, next to the reference's happo.yaml defaults; its tuned config.json files are in
tests/golden/reference_tuned_configs.json (both written by tests/golden/make_reference_configs.py).  This repo's
examples/train.py, which imports the same two names through the alias, must hand the runner the same three dicts.  The
runner class is replaced by a recorder (a real run needs a GPU; tests/test_gpu_iteration.py covers it)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
TRAIN = os.path.join(ROOT, "examples", "train.py")

OVERRIDES = ["--algo", "happo", "--env", "pettingzoo_mpe", "--exp_name", "alias", "--n_rollout_threads", "4096",
             "--continuous_actions", "False", "--lr", "0.001", "--hidden_sizes", "[64, 64]"]
TUNED_ALGOS = ["hatrpo", "haa2c", "mappo"]
TUNED_DIR = "pettingzoo_mpe/simple_spread_v2-continuous"   # tuned_configs/<env>/<scenario>/<algo>/config.json

DRIVER = r"""
import json, runpy, sys
sys.path.insert(0, {root!r})          # `harl` resolves to this repo's alias package
import harl, harl.runners
assert harl.__file__.startswith({root!r}), harl.__file__
calls = []
class Recorder:
    def __init__(self, args, algo_args, env_args):
        calls.append(dict(args=args, algo_args=algo_args, env_args=env_args))
    def run(self): calls[-1]["run"] = True
    def close(self): calls[-1]["close"] = True
for k in list(harl.runners.RUNNER_REGISTRY):
    harl.runners.RUNNER_REGISTRY[k] = Recorder
sys.argv = ["train.py"] + {argv!r}
runpy.run_path({train!r}, run_name="__main__")
print("RECORD " + json.dumps(calls))
"""


def record(train, argv, cwd):
    """Run the entry point ``train`` with ``argv`` against this package; the runner constructions it made."""
    code = DRIVER.format(root=ROOT, argv=argv, train=train)
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=cwd)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RECORD ")][-1]
    return json.loads(line[len("RECORD "):])


def _golden(name):
    with open(os.path.join(GOLDEN, name), encoding="utf-8") as fh:
        return json.load(fh)


def test_reference_train_py_builds_the_runner_from_this_repos_configs(tmp_path):
    calls = record(TRAIN, OVERRIDES, str(tmp_path))
    assert len(calls) == 1 and calls[0].get("run") and calls[0].get("close")
    c = calls[0]
    assert c["args"]["algo"] == "happo" and c["args"]["env"] == "pettingzoo_mpe" and c["args"]["exp_name"] == "alias"
    assert c["algo_args"]["train"]["n_rollout_threads"] == 4096          # command-line overrides reached the leaves
    assert c["algo_args"]["model"]["lr"] == 0.001 and c["algo_args"]["model"]["hidden_sizes"] == [64, 64]
    assert c["env_args"]["continuous_actions"] is False
    gold = _golden("reference_train_py.json")
    # the defaults are the reference's own (harl/configs/algos_cfgs/happo.yaml), key for key
    for section, leaves in gold["happo_yaml"].items():
        assert set(leaves) == set(c["algo_args"][section]), section
        for k, v in leaves.items():
            if (section, k) not in (("train", "n_rollout_threads"), ("model", "lr"), ("model", "hidden_sizes")):
                assert c["algo_args"][section][k] == v, (section, k)
    # and the runner receives what the reference's train.py gave it for the same command line
    assert gold["overrides"]["argv"] == OVERRIDES
    assert calls == gold["overrides"]["calls"]


@pytest.mark.parametrize("algo", TUNED_ALGOS)
def test_reference_train_py_load_config_and_other_on_policy_algorithms(algo, tmp_path):
    blob = _golden("reference_tuned_configs.json")[f"{TUNED_DIR}/{algo}/config.json"]
    tuned = tmp_path / "config.json"
    tuned.write_text(json.dumps(blob), encoding="utf-8")
    calls = record(TRAIN, ["--load_config", str(tuned), "--exp_name", "tuned"], str(tmp_path))
    c = calls[0]
    assert c["args"]["algo"] == blob["main_args"]["algo"] == algo
    assert c["algo_args"] == blob["algo_args"] and c["env_args"] == blob["env_args"]
    ref = _golden("reference_train_py.json")["load_config"][algo]
    assert len(calls) == len(ref) == 1 and c["args"]["load_config"] == str(tuned)
    for key in ("algo_args", "env_args", "run", "close"):
        assert c[key] == ref[0][key], key
    assert {k: v for k, v in c["args"].items() if k != "load_config"} == \
        {k: v for k, v in ref[0]["args"].items() if k != "load_config"}
