"""hb_gae_returns variants at the C2 shape and 16x wider: microseconds per launch (bench.gae_microbench: CUDA-graph
replay over 8 rotating buffer sets > L2), next to a plain copy of the same bytes.  Run on the GPU box:
    python profiles/gae_variants.py > profiles/gae_variants_r02.txt"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CODE = """
import sys, json; sys.path.insert(0, %r)
import torch, bench
from harl_b200 import _lib as L
peaks = bench.load_peaks()
out = {}
for C in (4096, 65536):
    out[C] = bench.gae_microbench(torch, 200, C, peaks)
print(json.dumps(out))
""" % ROOT

print("# variant                          [200,4096] us  GB/s  copy us | [200,65536] us  GB/s  copy us")
for name, env in (("segmented, sequential carry", dict(HB_GAE_IMPL="1")),
                  ("segmented, parallel-scan carry", dict(HB_GAE_IMPL="2"))):
    r = subprocess.run([sys.executable, "-c", CODE], env={**os.environ, **env}, capture_output=True, text=True)
    if r.returncode != 0:
        print(name, "FAILED", r.stderr[-500:])
        continue
    o = json.loads(r.stdout.strip().splitlines()[-1])
    a, b = o["4096"], o["65536"]
    print(f"{name:32s} {a['avg_us']:8.2f} {a['achieved']:7.0f} {a['same_bytes_copy_us']:7.2f}  | "
          f"{b['avg_us']:8.2f} {b['achieved']:7.0f} {b['same_bytes_copy_us']:7.2f}")
