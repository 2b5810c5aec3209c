"""Sweep the CTA cap of the RNN weight-gradient GEMMs that run beside a recurrence (ops.wgrad_cta_cap) on the
flagship PlayLMP step: each setting runs bench.py in a fresh process with the rule replaced, and prints its ms_per_step.

    python scripts/wgrad_cap_sweep.py [--steps 200] [--repeats 5]

Settings alternate within each repeat, so drift of the card affects all of them alike.

A setting maps the lane count of the concurrent recurrence (1 or 2) to a cap; "rule" is ops.wgrad_cta_cap."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SETTINGS = {"rule": None, "1:64,2:20": {1: 64, 2: 20}, "1:42,2:20": {1: 42, 2: 20}, "1:84,2:10": {1: 84, 2: 10}}
RUN = """
import runpy, sys
sys.path.insert(0, {root!r})
from tacorl_b200 import ops
caps = {caps!r}
if caps is not None:
    ops.wgrad_cta_cap = lambda lanes: caps.get(lanes, 148)
sys.argv = ["bench.py"] + {args!r}
runpy.run_path({bench!r}, run_name="__main__")
"""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=5)
    a = ap.parse_args()
    args = ["--gpus", "1", "--steps", str(a.steps), "--warmup", "20", "--no-cpu-baseline", "--no-fp32", "--no-tacorl"]
    res = {}
    for _ in range(a.repeats):
        for name, caps in SETTINGS.items():
            code = RUN.format(root=ROOT, caps=caps, args=args, bench=os.path.join(ROOT, "bench.py"))
            out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT).stdout
            line = json.loads(out.strip().splitlines()[-1])
            res.setdefault(name, []).append(line["ms_per_step"])
            print(name, line["ms_per_step"], flush=True)
    for name, v in res.items():
        print(f"{name:14s} median {statistics.median(v):.4f} ms  min {min(v):.4f}  max {max(v):.4f}")


if __name__ == "__main__":
    main()
