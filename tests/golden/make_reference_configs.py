"""Write the reference data of tests/test_reference_entry_point.py and tests/test_tuned_configs.py from a checkout of
the unmodified reference (PKU-MARL/HARL):

    python tests/golden/make_reference_configs.py <reference checkout>

reference_tuned_configs.json  every on-policy tuned_configs/<env>/<scenario>/<algo>/config.json, keyed by its path below
                              tuned_configs/
reference_train_py.json       harl/configs/algos_cfgs/happo.yaml as parsed, and the (args, algo_args, env_args) that the
                              reference's examples/train.py hands to the runner for the command lines of the tests, run
                              against this package through the `harl` alias

Only configuration data and what the reference's code produced are stored, none of its code.
"""
import glob
import json
import os
import sys
import tempfile

import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from tests.test_reference_entry_point import OVERRIDES, TUNED_ALGOS, TUNED_DIR, record  # noqa: E402

ON_POLICY = ("happo", "hatrpo", "haa2c", "mappo")


def main(ref):
    tuned_root = os.path.join(ref, "tuned_configs")
    tuned = {}
    for f in sorted(glob.glob(os.path.join(tuned_root, "*", "*", "*", "config.json"))):
        with open(f, encoding="utf-8") as fh:
            blob = json.load(fh)
        if blob["main_args"]["algo"] in ON_POLICY:
            tuned[os.path.relpath(f, tuned_root).replace(os.sep, "/")] = blob
    with open(os.path.join(HERE, "reference_tuned_configs.json"), "w", encoding="utf-8") as fh:
        fh.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v, sort_keys=True)}" for k, v in tuned.items()) + "\n}\n")

    train = os.path.join(ref, "examples", "train.py")
    with open(os.path.join(ref, "harl", "configs", "algos_cfgs", "happo.yaml"), encoding="utf-8") as fh:
        out = dict(happo_yaml=yaml.safe_load(fh), load_config={})
    with tempfile.TemporaryDirectory() as tmp:
        out["overrides"] = dict(argv=OVERRIDES, calls=record(train, OVERRIDES, tmp))
        for algo in TUNED_ALGOS:
            with open(os.path.join(tmp, "config.json"), "w", encoding="utf-8") as fh:
                json.dump(tuned[f"{TUNED_DIR}/{algo}/config.json"], fh)
            out["load_config"][algo] = record(train, ["--load_config", "config.json", "--exp_name", "tuned"], tmp)
    with open(os.path.join(HERE, "reference_train_py.json"), "w", encoding="utf-8") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write("\n")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
