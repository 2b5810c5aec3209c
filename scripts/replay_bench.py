#!/usr/bin/env python
"""Training step fed from an HBM-resident replay (tacorl_b200.replay.DeviceReplay) next to the resident and host-fed
("e2e") steps of bench.py, in one process per GPU.

    python scripts/replay_bench.py --workload play_lmp|tacorl|cql_flat [--gpus N] --steps K --out DIR

Writes DIR/replay_bench_<workload>_n<N>.json (rank 0) with, per workload:
  replay   ms per step and frames/s with every batch sampled and assembled on the device inside the step's CUDA graph;
  resident / e2e   bench.py's measure_workload in the same process: batch resident in HBM / pinned host batch copied
           every step;
  sample_assembly  the sampler + gather launches alone (a CUDA graph of 20 sample() calls, CUDA events), the bytes they
           move (computed from shapes: every output byte read once from the store and written once) and the GB/s;
  device   name and power limit of the GPU.
The dataset is synthetic: per rank, `--episodes` episodes of `--episode-len` random 200x200 frames (several times the
126 MB L2), drawn with a seed of its own.  `--gpus N > 1` relaunches the script under torch.distributed.run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

KIND = {"play_lmp": "play_lmp", "tacorl": "tacorl", "cql_flat": "cql"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", required=True, choices=sorted(KIND))
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64, help="windows (transitions for cql_flat) per GPU")
    ap.add_argument("--episodes", type=int, default=64)
    ap.add_argument("--episode-len", type=int, default=64)
    ap.add_argument("--pad", type=int, default=6, help="RandomShiftsAug pad (0: no shift)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


def device_info(local):
    info = {"name": torch.cuda.get_device_name(local)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except Exception as e:  # pragma: no cover
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e!r}"
    return info


def synthetic_index(args, rank, hw):
    from tacorl_b200.replay import ReplayIndex
    g = np.random.default_rng(1000 + rank)
    eps = []
    for _ in range(args.episodes):
        n = args.episode_len
        act = g.uniform(-1, 1, (n, 7)).astype(np.float32)
        act[:, -1] = np.where(act[:, -1] > 0, 1.0, -1.0)
        eps.append({"rgb_static": g.integers(0, 256, (n, hw, hw, 3), dtype=np.uint8), "rel_actions": act})
    return ReplayIndex(eps)


def main():
    args = parse()
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr=127.0.0.1", "--master-port=29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    import bench
    from tacorl_b200 import _lib, runtime
    from tacorl_b200.replay import DeviceReplay

    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    ns = argparse.Namespace(gpus=args.gpus, steps=args.steps, warmup=args.warmup, batch=args.batch, scaling="weak",
                            global_batch=args.batch * args.gpus, workload=args.workload, input="u8", no_graph=False,
                            timeline=None, precision=args.precision)
    ctx = bench.Ctx(ns)
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    if world > 1:
        from tacorl_b200.parallel import collective_channels
        os.environ.setdefault("NCCL_MAX_NCHANNELS", str(collective_channels(world)))
        os.environ.setdefault("NCCL_MIN_NCHANNELS", str(collective_channels(world)))
        ctx.dist.init_process_group("nccl", device_id=dev)
        ctx.barrier()
    wl = bench.WORKLOADS[args.workload]
    B = args.batch
    frames_per = bench.frames_per_window(wl)

    # 1. resident and host-fed steps, exactly as bench.py measures them
    res, h = bench.measure_workload(ctx, args.workload, args.precision, args.steps, args.warmup)
    del h
    ctx.graphs.clear()
    torch.cuda.empty_cache()

    # 2. the same step fed from a DeviceReplay inside its graph
    m, opts, step_fn = bench.build_ours(wl, dev, world, args.precision)
    index = synthetic_index(args, rank, bench.IMG)
    kind = KIND[args.workload]
    replay = DeviceReplay(index, B, kind=kind, min_window=bench.T_FRAMES // 2, max_window=bench.T_FRAMES, pad=args.pad,
                          seed=12345 + rank, device=dev)
    graphed = runtime.GraphedTrainStep(step_fn, None, device=dev, warmup=3, source=replay)
    ctx.graphs.append(graphed)
    for _ in range(args.warmup):
        graphed()
    r0 = graphed.replays
    n0 = _lib.launch_count()
    ms = ctx.timed(lambda s: graphed(), args.steps) / args.steps
    launches = _lib.launch_count() - n0 + graphed.launches_per_replay * (graphed.replays - r0)
    loss = graphed.out
    final_loss = float(loss) if torch.is_tensor(loss) else None

    # 3. sampler + assembly alone: a graph of 20 sample() calls
    reps = 20
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        replay.sample()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            replay.sample()
    g.replay()
    torch.cuda.synchronize(dev)
    times = []
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        times.append(e0.elapsed_time(e1) / reps)
    sa_ms = float(np.median(times))
    out_bytes = replay.output_bytes
    moved = 2 * out_bytes                  # every output byte read once from the store, written once

    line = {"workload": args.workload, "n_gpus": world, "windows_per_gpu": B, "frames_per_window": frames_per,
            "precision": args.precision, "steps": args.steps, "warmup": args.warmup, "pad": args.pad,
            "dataset_per_rank": {"frames": index.num_frames, "bytes": index.nbytes,
                                 "episodes": args.episodes, "episode_len": args.episode_len},
            "replay": {"ms_per_step": ms, "frames_per_s": world * B * frames_per / (ms / 1e3),
                       "launches_per_step": launches / args.steps, "launches_per_replay": graphed.launches_per_replay,
                       "h2d_bytes_per_step": 0, "final_loss": final_loss},
            "resident": {"ms_per_step": res["ms_per_step"], "frames_per_s": res["value"],
                         "launches_per_step": res["launches_per_step"]},
            "e2e": {"ms_per_step": res["e2e"]["ms_per_step"], "frames_per_s": res["e2e"]["value"],
                    "h2d_bytes_per_step": res["e2e"]["h2d_bytes_per_step"]},
            "sample_assembly": {"ms": sa_ms, "bytes": moved, "gbs": moved / (sa_ms / 1e3) / 1e9,
                                "timing": f"CUDA events around a graph of {reps} sample() calls, median of 10"},
            "device": device_info(ctx.local)}
    line["replay_minus_resident_ms"] = ms - res["ms_per_step"]
    if rank == 0:
        os.makedirs(args.out, exist_ok=True)
        path = os.path.join(args.out, f"replay_bench_{args.workload}_n{world}.json")
        json.dump(line, open(path, "w"), indent=1)
        print(json.dumps(line), flush=True)
    del g
    bench.teardown(ctx)


if __name__ == "__main__":
    main()
