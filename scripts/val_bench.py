#!/usr/bin/env python
"""Validation sweeps (Trainer.validate over a DeviceReplay(mode="sweep")) at bench.py's sizes, one GPU.

    python scripts/val_bench.py --workload play_lmp|tacorl|cql_flat|all --out DIR

Writes DIR/val_bench_<workload>.json with, per workload (64 windows of 16 frames of 200x200, bf16 by default):
  graphed_batch_ms   one full validation batch replayed from the validation graph (sweep + gather + forward +
                     accumulate), CUDA events around --steps replays;
  eager_host_ms      one eager validation_step on a pinned host batch copied to the device: what a user without the
                     sweep runs, CUDA events around --steps calls;
  sweep_ms           one whole Trainer.validate over a synthetic split of --episodes x --episode-len frames (several
                     times the 126 MB L2), host clock around the call (it ends with the read-back), median of 5;
  graph_pool_bytes   device memory reserved by the first validate (validation graph capture and its pool);
  train_ms_without / train_ms_with   the replay-fed training step, CUDA events around --steps replays, timed before
                     any validation graph exists and again with one held, alternated --repeats times;
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

KIND = {"play_lmp": "play_lmp", "tacorl": "tacorl", "cql_flat": "cql"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", required=True, choices=sorted(KIND) + ["all"])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--episodes", type=int, default=48)
    ap.add_argument("--episode-len", type=int, default=64)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0 or args.repeats < 1:
        ap.error("--steps and --repeats must be at least 1, --warmup at least 0")
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


def pinned(batch):
    return {k: pinned(v) if isinstance(v, dict) else v.cpu().pin_memory() for k, v in batch.items()}


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
    val = DeviceReplay(index, B, kind=kind, min_window=bench.T_FRAMES // 2, max_window=bench.T_FRAMES, seed=777,
                       device=dev, mode="sweep")
    train_step = runtime.GraphedTrainStep(step_fn, None, device=dev, warmup=3, source=train)
    for _ in range(args.warmup):
        train_step()
    without = [events_ms(train_step, args.steps)]

    tr = TR.Trainer(precision=args.precision, device=dev)
    torch.cuda.synchronize()
    reserved0 = torch.cuda.memory_reserved(dev)
    tr.validate(m, val)
    torch.cuda.synchronize()
    pool = torch.cuda.memory_reserved(dev) - reserved0
    graph = tr._val_states[(id(m), id(val))]["graph"]
    m.train()

    with_val = []
    for r in range(args.repeats):
        with_val.append(events_ms(train_step, args.steps))
        if r + 1 < args.repeats:
            without.append(events_ms(train_step, args.steps))

    sweeps = []
    for _ in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        metrics = tr.validate(m, val)[0]
        sweeps.append((time.perf_counter() - t0) * 1e3)

    m.eval()
    val.reset()
    for _ in range(args.warmup):
        graph()
    graphed_ms = events_ms(graph, args.steps)
    val.reset()
    host = pinned(val.sample())

    def eager():
        with torch.no_grad():
            m.validation_step(TR._to_device(host, dev), 0)
    for _ in range(args.warmup):
        eager()
    eager_ms = events_ms(eager, args.steps)
    m.train()
    del graph
    return {"workload": workload, "precision": args.precision, "windows_per_batch": B,
            "frames_per_window": bench.frames_per_window(wl),
            "split": {"frames": index.num_frames, "bytes": index.nbytes, "items": val.items,
                      "batches_per_sweep": val.batches_per_sweep, "tail": val.tail},
            "graphed_batch_ms": graphed_ms, "eager_host_ms": eager_ms,
            "sweep_ms_median": float(np.median(sweeps)), "sweep_ms": sweeps, "graph_pool_bytes": int(pool),
            "launches_per_graphed_batch": tr._val_states[(id(m), id(val))]["graph"].launches_per_replay,
            "train_ms_without": without, "train_ms_with": with_val,
            "metrics": metrics, "device": device_info(0)}


def main():
    args = parse()
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    os.makedirs(args.out, exist_ok=True)
    for w in (sorted(KIND) if args.workload == "all" else [args.workload]):
        line = measure(args, w)
        with open(os.path.join(args.out, f"val_bench_{w}.json"), "w") as f:
            json.dump(line, f, indent=1)
        print(json.dumps(line), flush=True)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
