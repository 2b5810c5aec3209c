#!/usr/bin/env python
"""Cost of the critic-guided plan search (tacorl_b200.rollout.PlanSearch) in the rollout policy's replan step, bf16.

    python scripts/plan_search_bench.py --out DIR [--steps 200] [--warmup 20]

For n_envs in {1, 8, 64}, samples K in {64, 256} and iterations I in {1, 3} (elites K / 8, min_std 1e-3), on the
single-view TACO-RL agent (static 200x200, latent 16, decoder hidden 2048, critics 3 x 256, no optimiser: the eval
case, critic weights staged to bf16 inside the graph), writes DIR/plan_search_bench.json with, per n_envs:
  replan_step_ms      the replan step without the search (every row replanning; one CUDA-graph replay), CUDA events
                      over --steps steps;
  step_ms             the plain step (no replan), for scale;
and per (K, I): search_replan_step_ms, the same replan step with the search, and the library launches of its graph;
plus the device name and power limit, read in the same run.  Weights and inputs are synthetic (seeded)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from rollout_bench import build, device_info, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--envs", default="1,8,64")
    ap.add_argument("--samples", default="64,256")
    ap.add_argument("--iterations", default="1,3")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("plan_search_bench needs a CUDA device")
    from oracle import synth as S
    from tacorl_b200 import ops
    from tacorl_b200.rollout import PlanSearch, RolloutPolicy
    ops.set_precision("bf16")
    m = build(("rgb_static",), 16, 2048)
    res = {"device": device_info(), "precision": "bf16", "steps": args.steps, "warmup": args.warmup, "rows": []}
    for n in [int(v) for v in args.envs.split(",")]:
        goal = {"rgb_static": S.synth_images((n, 3, 200, 200), 1, "goal").cuda()}
        obs = {"rgb_static": S.synth_images((n, 3, 200, 200), 1, "obs").cuda()}

        def policy(search):
            pol = RolloutPolicy(m, n, seed=0, plan_search=search)
            pol.reset(list(range(n)), goal)
            pol.step(obs)
            return pol

        def replan_of(pol):
            def replan_step():
                pol.replan(list(range(n)))
                pol.step()
            return replan_step

        base = policy(None)
        row = {"n_envs": n, "replan_step_ms": timed(replan_of(base), args.steps, args.warmup),
               "step_ms": timed(base.step, args.steps, args.warmup), "search": []}
        for K in [int(v) for v in args.samples.split(",")]:
            for iters in [int(v) for v in args.iterations.split(",")]:
                pol = policy(PlanSearch(samples=K, elites=K // 8, iterations=iters, min_std=1e-3))
                ms = timed(replan_of(pol), args.steps, args.warmup)
                row["search"].append({"samples": K, "elites": K // 8, "iterations": iters,
                                      "search_replan_step_ms": ms, "launches": pol.launches[(True, "bf16")]})
                del pol
        res["rows"].append(row)
        print(json.dumps(row), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "plan_search_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["device"]))


if __name__ == "__main__":
    main()
