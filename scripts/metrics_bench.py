#!/usr/bin/env python
"""Cost of recording every training step's logged scalars (runtime.TrainMetricsRecorder) at bench.py's sizes, one GPU.

    python scripts/metrics_bench.py --workload play_lmp|tacorl|all --out DIR

Writes DIR/metrics_bench_<workload>.json with, per workload (64 windows of 16 frames of 200x200, bf16 by default,
replay-fed):
  train_ms_without / train_ms_with   the replay-fed step replayed from a plain GraphedTrainStep, and from one whose step
                     ends with the record launch followed by the Trainer's host-side step_done (ring read-back every
                     --log-every steps), CUDA events around --steps steps; the two graphs train the same module and are
                     timed alternately, --repeats times each;
  record_us          device time of one record launch: CUDA events around a graph of 200 record launches;
  readback_host_us   host time of a step_done that finishes a half (all-reduce skipped on one GPU, event, side-stream
                     copy to pinned memory, read of the previous copy), median; step_done_host_us: one that does not;
  launches_without / launches_with   library launches per replay;
  device             name and power limit of the GPU."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

KIND = {"play_lmp": "play_lmp", "tacorl": "tacorl"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", required=True, choices=sorted(KIND) + ["all"])
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--log-every", type=int, default=50)
    ap.add_argument("--episodes", type=int, default=48)
    ap.add_argument("--episode-len", type=int, default=64)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0 or args.repeats < 1 or args.log_every < 1:
        ap.error("--steps, --repeats and --log-every must be at least 1, --warmup at least 0")
    return args


def events_ms(fn, n):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def measure(args, workload):
    import bench
    from replay_bench import device_info, synthetic_index
    from tacorl_b200 import runtime
    from tacorl_b200 import trainer as TR
    from tacorl_b200.replay import DeviceReplay
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    wl = bench.WORKLOADS[workload]
    kind, B = KIND[workload], args.batch
    m, opts, step_fn = bench.build_ours(wl, dev, 1, args.precision)
    index = synthetic_index(args, 0, bench.IMG)
    train = DeviceReplay(index, B, kind=kind, min_window=bench.T_FRAMES // 2, max_window=bench.T_FRAMES, pad=6,
                         seed=12345, device=dev)
    plain = runtime.GraphedTrainStep(step_fn, None, device=dev, warmup=3, source=train)
    rec = runtime.TrainMetricsRecorder(dev, 2 * args.log_every, log_every_n_steps=args.log_every)
    recorded = runtime.GraphedTrainStep(TR._recording(step_fn, m, rec), None, device=dev, warmup=3, source=train)
    state = {"step": 0, "readback": [], "other": []}

    def with_recorder():
        recorded()
        t0 = time.perf_counter()
        rec.step_done(state["step"], 0)
        dt = (time.perf_counter() - t0) * 1e6
        state["step"] += 1
        state["readback" if state["step"] % args.log_every == 0 else "other"].append(dt)

    for _ in range(args.warmup):
        plain()
        with_recorder()
    without, with_rec = [], []
    for _ in range(args.repeats):
        without.append(events_ms(plain, args.steps))
        with_rec.append(events_ms(with_recorder, args.steps))
    rec.flush()

    g = torch.cuda.CUDAGraph()
    logged = {k: v for k, v in m.logged.items() if k.startswith("train/")}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        rec.record(logged)
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(g):
        for _ in range(200):
            rec.record(logged)
    g.replay()
    record_us = events_ms(g.replay, 20) / 200 * 1e3
    return {"workload": workload, "precision": args.precision, "windows_per_batch": B,
            "frames_per_window": bench.frames_per_window(wl), "log_every_n_steps": args.log_every,
            "keys": list(rec.keys), "steps_recorded": len(rec.history),
            "train_ms_without": without, "train_ms_with": with_rec,
            "train_ms_without_median": float(np.median(without)), "train_ms_with_median": float(np.median(with_rec)),
            "record_us": record_us, "readback_host_us": float(np.median(state["readback"])),
            "step_done_host_us": float(np.median(state["other"])),
            "launches_without": plain.launches_per_replay, "launches_with": recorded.launches_per_replay,
            "device": device_info(0)}


def main():
    args = parse()
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    os.makedirs(args.out, exist_ok=True)
    for w in (sorted(KIND) if args.workload == "all" else [args.workload]):
        line = measure(args, w)
        with open(os.path.join(args.out, f"metrics_bench_{w}.json"), "w") as f:
            json.dump(line, f, indent=1)
        print(json.dumps(line), flush=True)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
