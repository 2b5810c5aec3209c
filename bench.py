#!/usr/bin/env python
"""bench.py — PlayLMP + TACO-RL training-step throughput on N B200s, one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload play_lmp|tacorl|play_lmp_multiview|tacorl_multiview]
                    [--precision bf16|fp32] [--scaling weak|strong] [--batch 64] [--global-batch 512]
                    [--dump-outputs DIR]

Metric (BASELINE.json): train frames/sec.  A step = one optimiser step (forward + backward + gradient all-reduce +
Adam[s]) on a synthetic CALVIN-shaped batch of windows x 16 frames of 3x200x200 per GPU.  The headline line is the
PlayLMP step (BASELINE configs[1]); the TACO-RL step (configs[2]) is measured with the same rules and rides in the
`tacorl` object of the same line (`--workload tacorl` makes it the line itself; `*_multiview` = configs[3]).
`--scaling weak` (default): `--batch` windows per GPU; `--scaling strong`: `--global-batch` windows split over the
ranks (configs[4]).  `value` is timed with inputs resident in HBM; `e2e` re-times the same steps through the public
module API with the batch in pinned host memory (H2D copy of every step's inputs and a D2H read of its loss inside
the timed region).

`--impl reference` times the UNMODIFIED reference modules (imported from oracle/_ref, the tree
oracle/vendor_reference.py copies from /root/reference; the oracle port when that tree is absent) on the host
cores, same workload, and -- when a GPU is visible -- the same reference modules under torch eager on the B200
(fp32 with TF32 convolutions, and bf16 autocast): the honest bar next to the CPU number.
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

T_FRAMES, IMG, GRIP = 16, 200, 84
# ---- algorithmic work (SURVEY.md section 8(d); de-duplicated minimum of a correct implementation)
ENC_FLOP_PER_FRAME = 260.8e6            # encoder fwd+bwd per 200x200 frame (96.8 fwd + 164.0 bwd)
ENC_FLOP_PER_FRAME_84 = 36.8e6          # 84x84 gripper view
# Algorithmic HBM bytes of the encoder fwd+bwd per 200x200 frame, SURVEY 8(d): uint8 input read by conv1 forward and by
# its weight gradient 2 x 120000; bf16 saved activations y1 153664 + y2 67712 + y3 56448 written once, read once.
ENC_BYTES_PER_FRAME = 2 * 120_000 + 2 * (153_664 + 67_712 + 56_448)        # 795 648
# What this implementation must move on top of that (DESIGN.md section 4): the gradient maps dy1/dy2/dy3 (written once,
# read by the data- and weight-gradient kernels), y3 kept in fp32 for the soft-argmax: 2 144 000 B per frame.
ENC_BYTES_PER_FRAME_IMPL = 2_144_000
# dram__bytes_read.sum + dram__bytes_write.sum over every launch of one encoder forward+backward pass under ncu
# (scripts/profile_encoder.py, 1024 frames; profiles/r02_launches_summary.md section 4, final state of round 2: 3255 MB with
# float frames - 368 MB the uint8 s2d does not read = 2887 MB; round 1 measured 2837 MB, profiles/r01_encoder_kernels_ncu.md)
ENC_NCU_TRAFFIC_BYTES = 2.887e9
PLAYLMP_FLOP_PER_WINDOW = 8.97e9        # BiRNN recogniser, 16 x 200x200 frames
TACORL_FLOP_PER_WINDOW = 5.89e9         # 27 encoder fwd + 6 bwd frames, PR fwd, decoder fwd+bwd, MLPs
RNN_H = 2048
DUMP_SAMPLE = 32768                 # --dump-outputs: elements kept per tensor
DUMP_MAX_BYTES = 64 << 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("TACORL_PRECISION", "bf16"), choices=["fp32", "bf16"])
    ap.add_argument("--batch", type=int, default=64, help="windows per GPU (weak scaling)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--global-batch", type=int, default=512, help="windows per step over all GPUs (strong scaling)")
    ap.add_argument("--workload", default="play_lmp",
                    choices=["play_lmp", "tacorl", "play_lmp_multiview", "tacorl_multiview", "cql_flat"])
    ap.add_argument("--input", default="u8", choices=["u8", "f32"],
                    help="frame dtype fed to the step: u8 = raw uint8 frames, scale+normalise fused on the device; "
                         "f32 = pre-normalised float32 (the reference DataLoader's output)")
    ap.add_argument("--no-tacorl", action="store_true", help="skip the TACO-RL object of the PlayLMP line")
    ap.add_argument("--no-fp32", action="store_true", help="skip the short fp32-path measurement of the PlayLMP line")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--timeline", default=None,
                    help="after the measurement, record the kernel timeline of ONE more graph replay (CUPTI through "
                         "torch.profiler, every rank replays, rank 0 writes this JSON file): for shares and gaps only")
    ap.add_argument("--no-gpu-eager", action="store_true", help="reference arm: skip the torch-eager-on-GPU timings")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--cpu-steps", type=int, default=3, help="timed steps of the cpu_baseline leg of our own line")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps of the headline workload, write what its last step computed as "
                         "DIR/<name>.npy (float32): the returned loss, the logged scalars, every floating-point "
                         "state_dict entry after the update and every parameter's gradient; a tensor of more than "
                         f"{DUMP_SAMPLE} elements is stored as a fixed, seeded sample of its flattened elements")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def dump_outputs(out_dir, loss, module, opts):
    """Writes the outputs of the last timed step (see --dump-outputs).  Inputs, initial weights and noise are seeded, so
    two builds run with the same arguments can be compared file for file."""
    import numpy as np
    names = {id(p): n for n, p in module.named_parameters()}
    arrays = {"loss": loss}
    arrays.update({"logged." + k.replace("/", "."): v for k, v in module.logged.items() if torch.is_tensor(v)})
    arrays.update({"state." + k: v for k, v in module.state_dict().items() if v.dtype.is_floating_point})
    for o in opts:
        for p, g in zip(o.param_groups[0]["params"], o.grad_views):
            arrays["grad." + names[id(p)]] = g
    total = sum(4 * min(t.numel(), DUMP_SAMPLE) for t in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the limit of {DUMP_MAX_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if a.numel() > DUMP_SAMPLE:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE]
            a = a.reshape(-1)[idx.sort().values]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def windows_per_gpu(args, world):
    if args.scaling == "strong":
        assert args.global_batch % world == 0, "--global-batch must divide over the ranks"
        return args.global_batch // world
    return args.batch


# ----------------------------------------------------------------------------------- workloads
WORKLOADS = {
    "play_lmp": dict(module="play_lmp", mods=("rgb_static",), goal_mods=("rgb_static",), latent=16,
                     desc="PlayLMP[BiRNN tanh_net] train step (fwd+bwd+allreduce+Adam), static 3x200x200, 16 frames/window, "
                          "BASELINE configs[1]", metric="play_lmp_train_frames_per_sec", flop=PLAYLMP_FLOP_PER_WINDOW),
    "tacorl": dict(module="tacorl", mods=("rgb_static",), goal_mods=("rgb_static",), latent=16,
                   desc="TACORL[BiRNN PR] train step: frozen LMP encode (16 frames) + decoder finetune + CQL update "
                        "(n_action_samples 4, Lagrange, BC epoch) + Polyak, static 3x200x200 + goal image, BASELINE configs[2]",
                   metric="tacorl_train_frames_per_sec", flop=TACORL_FLOP_PER_WINDOW),
    "play_lmp_multiview": dict(module="play_lmp", mods=("rgb_static", "rgb_gripper"), goal_mods=("rgb_static", "rgb_gripper"),
                               latent=32, desc="PlayLMP[BiRNN] train step, static 3x200x200 + gripper 3x84x84 views, latent "
                               "plan 32 (play_lmp_gripper_real_world), BASELINE configs[3]",
                               metric="play_lmp_multiview_train_frames_per_sec",
                               flop=PLAYLMP_FLOP_PER_WINDOW + 16 * ENC_FLOP_PER_FRAME_84),
    "tacorl_multiview": dict(module="tacorl", mods=("rgb_static", "rgb_gripper"), goal_mods=("rgb_static", "rgb_gripper"),
                             latent=32, desc="TACORL train step on a multi-view LMP (tacorl_real_world): static 3x200x200 + "
                             "gripper 3x84x84 for observation and goal, latent plan 32, BASELINE configs[3]",
                             metric="tacorl_multiview_train_frames_per_sec",
                             flop=TACORL_FLOP_PER_WINDOW + (27 * 13.9e6 + 6 * 22.9e6)),
    # SURVEY 8f-4: the paper's flat baseline.  A "window" is one transition = 3 frames (observation, next, goal);
    # 11 encoder forwards (actor: obs+goal, next; q1, q2: obs+goal; targets: next+goal) + 6 backward frames per transition
    "cql_flat": dict(module="cql", mods=("rgb_static",), goal_mods=("rgb_static",), latent=16, frames=3,
                     desc="flat CQL_Offline baseline (cql_offline_goal_cond / cql_real_world): discrete-gripper actor, "
                          "twin visual critics, entropy-regularised backup, Lagrange, n_action_samples 4, BC epoch; "
                          "one transition = observation + next observation + goal image, static 3x200x200",
                     metric="cql_flat_train_frames_per_sec", flop=(11 * 96.8e6 + 6 * 164e6)),
}


def frames_per_window(wl):
    return wl.get("frames", T_FRAMES)


def host_batch(wl, B, seed, u8):
    """Synthetic CALVIN-shaped batch in pinned host memory (SURVEY 8(d) "Synthetic inputs")."""
    from tacorl_b200.utils import synthetic
    if wl["module"] == "cql":
        return cql_host_batch(B, seed, u8)
    b = synthetic.play_batch(B, T_FRAMES, IMG, IMG, seed=seed, with_goal=(wl["module"] == "tacorl"),
                             modalities=wl["mods"], goal_modalities=wl["goal_mods"], gripper_hw=(GRIP, GRIP))
    out = {"states": dict(b["states"]), "actions": b["actions"]}
    if wl["module"] == "tacorl":
        out["goal"], out["disp"] = dict(b["goal"]), b["disp"]

    def conv(t):
        if u8:      # raw frames; (u8/255 - 0.5)/0.5 happens inside the first encoder kernel
            t = ((t + 1.0) * 127.5).round().clamp(0, 255).to(torch.uint8)
        return t.pin_memory()

    out["states"] = {k: conv(v) for k, v in out["states"].items()}
    if "goal" in out:
        out["goal"] = {k: conv(v) for k, v in out["goal"].items()}
    out["actions"] = out["actions"].pin_memory()
    if "disp" in out:
        out["disp"] = out["disp"].pin_memory()
    return out


def cql_host_batch(B, seed, u8):
    """Transition batch of GoalCondReplayBufferDataset.get_transition (goal_cond_replay_buffer_dataset.py:277-296) in
    pinned host memory."""
    g = torch.Generator().manual_seed(seed)

    def img():
        t = torch.randint(0, 256, (B, 3, IMG, IMG), generator=g, dtype=torch.uint8)
        return (t if u8 else t.float() / 127.5 - 1.0).pin_memory()

    obs, nxt, goal = {"rgb_static": img()}, {"rgb_static": img()}, {"rgb_static": img()}
    actions = torch.rand(B, 7, generator=g) * 2 - 1
    actions[:, -1] = torch.where(actions[:, -1] > 0, 1.0, -1.0)
    hit = (torch.rand(B, generator=g) < 0.3).long()
    return {"observations": {"observation": obs, "goal": goal}, "actions": actions.pin_memory(),
            "next_observations": {"observation": nxt, "goal": goal}, "rewards": hit.clone().pin_memory(),
            "terminals": hit.clone().pin_memory()}


def nbytes(batch):
    n = 0
    for v in batch.values():
        n += nbytes(v) if isinstance(v, dict) else v.numel() * v.element_size()
    return n


def to_device(batch, dev):
    return {k: (to_device(v, dev) if isinstance(v, dict) else v.to(dev, non_blocking=True)) for k, v in batch.items()}


def build_ours(wl, dev, world, precision):
    from tacorl_b200 import configs, ops, parallel, runtime
    from tacorl_b200.utils import synthetic
    from tacorl_b200.utils.config import instantiate
    ops.set_precision(precision)
    torch.manual_seed(0)
    if wl["module"] == "cql":
        m = instantiate(configs.cql_offline_goal_cond(wl["mods"], wl["goal_mods"]))
        synthetic.init_like_reference(m, seed=0)
        m.to(dev)
        m.train()
        opts = m.optimizers()
        if world > 1:
            for o in opts:
                parallel.attach_data_parallel(o, world)
        return m, opts, runtime.tacorl_step_fn(m)
    lmp = instantiate(configs.play_lmp_for_rl("tanh_net", modalities=wl["mods"], latent_plan_dim=wl["latent"],
                                              goal_modalities=wl["goal_mods"]))
    if wl["module"] == "play_lmp":
        m = lmp
        synthetic.init_like_reference(m, seed=0)          # identical random-init weights on every rank
        m.to(dev)
        opts = [m.configure_optimizers()]
        fn = runtime.play_lmp_step_fn(m, opts[0])
    else:
        m = instantiate(configs.tacorl(), play_lmp=lmp)
        synthetic.init_like_reference(m, seed=0)
        m.to(dev)
        opts = m.optimizers()
        fn = runtime.tacorl_step_fn(m)
    m.train()
    if world > 1:
        for o in opts:
            parallel.attach_data_parallel(o, world)
    return m, opts, fn


# ----------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock / throttle-reason samples DURING the timed region: an NVML polling thread (a sample every few ms; the
    timed region of a default run is only tens of ms long, too short for `nvidia-smi -lms`)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.samples, self.reasons, self.power = [], set(), []
        self._stop = None
        self._thread = None
        self.max_mhz = None
        self.err = None

    def _run(self, nv, h):
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1e3)
            except Exception as e:  # pragma: no cover
                self.err = repr(e)
                return
            time.sleep(0.002)

    def start(self):
        import threading
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and vis.split(",")[self.idx].isdigit() else self.idx
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            self._stop = threading.Event()
            self._thread = threading.Thread(target=self._run, args=(nv, h), daemon=True)
            self._thread.start()
        except Exception as e:
            self.err = repr(e)

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable: " + str(self.err)], "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_min_mhz": min(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples),
                "power_w_max": max(self.power) if self.power else None, "source": "nvml, sampled during the timed region"}


def trace(msg):
    if os.environ.get("BENCH_TRACE"):
        sys.stderr.write(f"[bench rank {os.environ.get('RANK', '0')} +{time.perf_counter():.1f}s] {msg}\n")
        sys.stderr.flush()


# ----------------------------------------------------------------------------------- our arm: one workload
class Ctx:
    """Process-wide pieces shared by every measurement of our arm."""

    def __init__(self, args):
        import torch.distributed as dist
        self.args = args
        self.dist = dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        # host threads and pinned staging buffers on the GPU's own NUMA node (every rank of a multi-GPU run pulls its
        # 123 MB batch from host memory each step; TACORL_NUMA_BIND=0 disables, =1 forces it for a single rank too)
        self.numa = {"bound": False, "why": "single rank"}
        want = os.environ.get("TACORL_NUMA_BIND")
        if want == "1" or (want is None and self.world > 1):
            from tacorl_b200.utils.numa import bind_to_gpu_node
            self.numa = bind_to_gpu_node(self.local)
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.graphs = []          # every captured graph, released before the process group is destroyed

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, n):
        """n calls of fn bracketed by barrier + synchronize, CUDA events on the launch stream, max over ranks (ms)."""
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(n):
            fn(s)
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms)


def measure_workload(ctx, name, precision, steps, warmup, e2e=True, sample_clocks=False, dump_dir=None):
    """Resident and end-to-end timing of one workload.  Returns (result dict, handles for the roofline probes).
    dump_dir: rank 0 writes the outputs of the last resident timed step there (dump_outputs)."""
    from tacorl_b200 import _lib, runtime
    args, dev, world, rank = ctx.args, ctx.dev, ctx.world, ctx.rank
    wl = WORKLOADS[name]
    B = windows_per_gpu(args, world)
    m, opts, eager_step = build_ours(wl, dev, world, precision)
    host = host_batch(wl, B, seed=1 + rank, u8=(args.input == "u8"))
    resident = to_device(host, dev)
    h2d = nbytes(host)
    graphed = None
    if not args.no_graph:
        graphed = runtime.GraphedTrainStep(eager_step, resident, device=dev, warmup=3, buffers=2)
        ctx.graphs.append(graphed)

    last = [None]

    def step(_s):
        last[0] = graphed() if graphed is not None else eager_step(resident)

    for s in range(warmup):
        step(s)
    clocks = ClockSampler(ctx.local) if (sample_clocks and rank == 0) else None
    if clocks:
        clocks.start()
    n0 = _lib.launch_count()
    r0 = graphed.replays if graphed is not None else 0
    total_ms = ctx.timed(step, steps)
    launches = _lib.launch_count() - n0
    if graphed is not None:     # replayed kernels: (kernels recorded in the graph) x (replays in the timed region)
        launches += graphed.launches_per_replay * (graphed.replays - r0)
    clk = clocks.stop() if clocks else None
    ms = total_ms / steps
    frames = world * B * frames_per_window(wl)
    res = {"metric": wl["metric"], "value": frames / (ms / 1e3), "unit": "frames/s", "ms_per_step": ms,
           "windows_per_sec": world * B / (ms / 1e3), "gpu_launches": launches, "launches_per_step": launches / steps,
           "cuda_graph": graphed is not None, "workload": wl["desc"],
           "algorithmic_tflops_whole_step": world * B * wl["flop"] / (ms / 1e3) / 1e12}
    if clk is not None:
        res["clocks"] = clk
    trace(f"{name}/{precision}: resident {ms:.3f} ms/step")
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, last[0], m, opts)
    if ctx.args.timeline and graphed is not None and name == ctx.args.workload:
        from torch.profiler import ProfilerActivity, profile
        ctx.barrier()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            graphed()
            torch.cuda.synchronize()
        ctx.barrier()
        if rank == 0:
            evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.time_range is not None]
            ks = sorted(((e.time_range.start, e.time_range.end, e.name) for e in evs), key=lambda t: t[0])
            t0 = ks[0][0] if ks else 0
            json.dump([{"start_us": a - t0, "dur_us": b - a, "name": n[:120]} for a, b, n in ks], open(ctx.args.timeline, "w"))

    if e2e:
        # end-to-end: pinned host batch -> H2D every step, loss read back every step.  With the graph runner the copy
        # of the next step's batch is issued on a copy stream while the current step runs (pinned-memory prefetch) and
        # the loss travels through an asynchronous D2H copy that the host reads one launch later; every timed step
        # still contains one full-batch H2D and one D2H read of its loss, and the last loss is read before the closing
        # event.  BENCH_E2E_SYNC=1: blocking float(loss) per step instead.
        losses = []
        if graphed is not None and os.environ.get("BENCH_E2E_SYNC", "") != "1":
            pinned = [torch.empty((), dtype=torch.float32, pin_memory=True) for _ in range(2)]
            done = [torch.cuda.Event() for _ in range(2)]
            stepped = [torch.cuda.Event() for _ in range(2)]
            rb = torch.cuda.Stream(device=dev)       # loss read-back stream: the main stream carries graph launches only
            main = torch.cuda.current_stream(dev)
            for e in done:
                e.record(main)

            def read(i):
                done[i % 2].synchronize()
                losses.append(float(pinned[i % 2]))

            def fn(s):
                main.wait_event(done[s % 2])         # (long complete) the slot's previous read-back, before its loss is rewritten
                loss = graphed()
                stepped[s % 2].record(main)
                with torch.cuda.stream(rb):
                    rb.wait_event(stepped[s % 2])
                    pinned[s % 2].copy_(loss, non_blocking=True)
                    done[s % 2].record(rb)
                if not os.environ.get("BENCH_E2E_NO_H2D"):        # (diagnostic knob: never set for a reported number)
                    graphed.prefetch(host)
                if s > 0:
                    read(s - 1)
                if s == steps - 1:
                    read(s)

            graphed.prefetch(host)
            graphed()                                # warm the staging path; leaves the next batch prefetched
            graphed.prefetch(host)
            torch.cuda.synchronize()
            e2e_ms = ctx.timed(fn, steps) / steps
            mode = "loss copied D2H asynchronously every step, read on the host one launch later"
        else:
            def fn(s):
                if graphed is not None:
                    loss = graphed()
                    graphed.prefetch(host)
                else:
                    loss = eager_step(to_device(host, dev))
                losses.append(float(loss))

            if graphed is not None:
                graphed.prefetch(host)
            fn(0)
            e2e_ms = ctx.timed(fn, steps) / steps
            mode = "synchronous loss read every step"
        res["e2e"] = {"value": frames / (e2e_ms / 1e3), "unit": "frames/s", "ms_per_step": e2e_ms,
                      "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "loss_read": mode,
                      "h2d_gbs_per_rank": h2d / (e2e_ms / 1e3) / 1e9, "numa": ctx.numa}
        res["final_loss"] = losses[-1] if losses else None
        trace(f"{name}/{precision}: e2e {e2e_ms:.3f} ms/step")
    return res, {"module": m, "opts": opts, "resident": resident, "B": B, "host": host}


# ----------------------------------------------------------------------------------- roofline probes
def roofline_encoder(ctx, h, ms_per_step, pk, pk_kind):
    """Vision encoder forward+backward (s2d + implicit-GEMM convs fwd/dgrad/wgrad + soft-argmax + FC) timed alone."""
    B = h["B"]
    enc = h["module"].perceptual_encoder.networks["rgb_static"]
    frames = h["resident"]["states"]["rgb_static"].view(B * T_FRAMES, 3, IMG, IMG)

    def enc_fb(_):
        for p in enc.parameters():
            p.grad = None
        e = enc(frames)
        e.backward(torch.ones_like(e))

    enc_fb(0)
    enc_ms = ctx.timed(enc_fb, 5) / 5
    n = B * T_FRAMES
    gbs = n * ENC_BYTES_PER_FRAME / (enc_ms / 1e3) / 1e9
    gbs_impl = n * ENC_BYTES_PER_FRAME_IMPL / (enc_ms / 1e3) / 1e9
    tf = n * ENC_FLOP_PER_FRAME / (enc_ms / 1e3) / 1e12
    # 260.8 MFLOP over 0.796 MB per frame = 328 FLOP/B, above the ridge of the measured peaks (1623 TF/s / 6.54 TB/s =
    # 248 FLOP/B) with SURVEY 8(d)'s bytes, below it (122 FLOP/B) with the gradient maps this implementation stores:
    # both fractions are reported; the HBM one is `frac`
    return {"kernel": "lmp_encoder fwd+bwd pass (s2d + implicit-GEMM convs fwd/dgrad/wgrad + soft-argmax + FC), timed alone",
            "bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "peak_kind": pk_kind + " burst (copy)", "unit": "GB/s",
            "frac": gbs / pk["hbm_gbs"],
            "traffic": ENC_NCU_TRAFFIC_BYTES * n / 1024 if ctx.args.input == "u8" else None,
            "algorithmic_bytes_per_launch": n * ENC_BYTES_PER_FRAME,
            "algorithmic_bytes_source": "SURVEY.md 8(d): uint8 input 2 x 120000 + bf16 saved activations 2 x 277824 per frame",
            "ms_per_launch": enc_ms, "share_of_step": enc_ms / ms_per_step,
            "with_gradient_maps": {"bytes_per_frame": ENC_BYTES_PER_FRAME_IMPL, "achieved": gbs_impl,
                                   "frac": gbs_impl / pk["hbm_gbs"]},
            "tensor": {"achieved": tf, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": tf / pk["bf16_tflops"],
                       "algorithmic_flops_per_launch": n * ENC_FLOP_PER_FRAME}}


def roofline_recurrence(ctx, h, ms_per_step, pk, pk_kind):
    """Action-decoder RNN (2 layers x 15 dependent steps, batch 2B: sampled + random plan) forward+backward alone."""
    from tacorl_b200 import ops
    B = h["B"]
    rnn = h["module"].action_decoder.rnn
    T, M, I = T_FRAMES - 1, 2 * B, rnn.input_size
    x = torch.randn(T, M, I, device=ctx.dev) * 0.1
    ws = rnn.weights()

    def fb(_):
        for p in ws:
            p.grad = None
        xx = x.clone().requires_grad_(True)
        out, _ = ops.relu_rnn(xx, ws, rnn.num_layers, False)
        out.backward(torch.ones_like(out) * 1e-3)

    fb(0)
    ms = ctx.timed(fb, 5) / 5
    H = RNN_H
    fwd = 2.0 * T * M * (I * H + H * H) + 2.0 * T * M * 2 * H * H          # input projections + recurrent products
    flops = 3.0 * fwd
    dep_steps = 4 * T                                                        # 2 layers x (forward + BPTT)
    tf = flops / (ms / 1e3) / 1e12
    step_flops = 2.0 * M * H * H
    return {"kernel": "action-decoder ReLU RNN forward+backward (rnn_seq / rnn_wave kernels + input / weight-gradient GEMMs), timed alone",
            "bound": "tensor", "achieved": tf, "peak": pk["bf16_tflops_sustained"], "peak_kind": pk_kind + " sustained (cuBLAS bf16)",
            "unit": "TFLOP/s", "frac": tf / pk["bf16_tflops_sustained"], "traffic": None,
            "algorithmic_flops_per_launch": flops, "ms_per_launch": ms, "share_of_step": None,
            "dependent_steps": dep_steps, "us_per_dependent_step": 1e3 * ms / dep_steps,
            "tflops_per_dependent_step": step_flops / (1e-3 * ms / dep_steps) / 1e12, "batch_rows": M}


def roofline_adam(ctx, h, pk, pk_kind):
    opt = h["opts"][0]
    n = opt.flat_params.numel()

    def st(_):
        opt.step(gathered=True)

    snap = opt.snapshot()
    st(0)
    ms = ctx.timed(st, 5) / 5
    opt.restore(snap)
    nb = n * (16 + 12 + (2 if opt.shadow is not None else 0))              # read p,g,m,v; write p,m,v (+ bf16 twin)
    gbs = nb / (ms / 1e3) / 1e9
    return {"kernel": "adam_kernel over the flat parameter buffer", "bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"],
            "peak_kind": pk_kind + " burst (copy)", "unit": "GB/s", "frac": gbs / pk["hbm_gbs"], "traffic": None,
            "algorithmic_bytes_per_launch": nb, "ms_per_launch": ms}


# ----------------------------------------------------------------------------------- reference modules (CPU / GPU eager)
def reference_kind():
    from oracle import ref_loader
    return "reference" if ref_loader.reference_available() else "port"


def reference_batch(wl, B, seed=1):
    from oracle import synth as S
    if wl["module"] == "cql":
        return S.synth_cql_batch(B, IMG, IMG, seed, modalities=wl["mods"], goal_modalities=wl["goal_mods"])
    return S.synth_play_batch(B, T_FRAMES, IMG, IMG, seed, modalities=wl["mods"], gripper_hw=(GRIP, GRIP),
                              with_goal=(wl["module"] == "tacorl"), goal_modalities=wl["goal_mods"])


def build_reference(wl, device="cpu"):
    """The unmodified reference module (+ its own torch.optim.Adam[s]) with the synthetic weights."""
    from oracle import ref_loader as R
    from oracle import synth as S
    torch.manual_seed(0)
    if wl["module"] == "cql":
        m = R.build_reference_cql(obs_modalities=list(wl["mods"]), goal_modalities=list(wl["goal_mods"]))
    else:
        lmp = R.build_reference_play_lmp(pr_kind="tanh_net", rnn_hidden=RNN_H, dropout_p=0.0, max_window=T_FRAMES,
                                         modalities=wl["mods"], goal_modalities=wl["goal_mods"],
                                         latent_plan_dim=wl["latent"])
        m = lmp if wl["module"] == "play_lmp" else R.build_reference_tacorl(lmp)
    shapes = {k: list(v.shape) for k, v in m.state_dict().items()}
    m.load_state_dict(S.synth_state_dict(shapes, 0))
    m.to(device)
    m.train()
    if wl["module"] == "play_lmp":
        opt = m.configure_optimizers()

        def step(batch, s):
            opt.zero_grad()
            loss = m.training_step(batch, s)
            loss.backward()
            opt.step()
            return loss
    else:
        m.optimizers()

        def step(batch, s):
            m.training_step(batch, s) if wl["module"] == "cql" else m.training_step(batch)
            return m.logged.get("train/q1_loss")
    return m, step


def port_step(wl, B):
    """Fallback when the reference tree did not travel: the oracle port of the same step."""
    from oracle import synth as S
    from oracle import tacorl_oracle as O
    from tests.gpu_util import build_cql_flat, build_play_lmp, build_tacorl
    if wl["module"] == "cql":
        m = build_cql_flat()
        shapes = {k: list(v.shape) for k, v in m.state_dict().items()}
        P = O.params_from(S.synth_state_dict(shapes, 0))
        opt = O.new_tacorl_opt_state(P)

        def step(batch, s):
            torch.manual_seed(1000 + s)
            return O.cql_training_step(P, opt, batch, O.draw_cql_noise(B), {}, 0)[0]["q1_loss"]
        return step
    lmp = build_play_lmp("tanh_net", wl["mods"], RNN_H, wl["latent"], T_FRAMES, goal_modalities=wl["goal_mods"])
    m = lmp if wl["module"] == "play_lmp" else build_tacorl(lmp)        # shapes only (no kernels run)
    shapes = {k: list(v.shape) for k, v in m.state_dict().items()}
    del m, lmp
    cfg = {"modalities": list(wl["mods"]), "goal_modalities": list(wl["goal_mods"]), "pr_kind": "tanh_net"}
    if wl["module"] == "play_lmp":
        P, opt = O.params_from(S.synth_state_dict(shapes, 0)), {}

        def step(batch, s):
            torch.manual_seed(1000 + s)
            noise = O.draw_play_lmp_noise(B, T_FRAMES, latent=wl["latent"], goal_dim=32 * len(wl["goal_mods"]))
            return O.play_lmp_training_step(P, opt, batch, noise, cfg)[0]["total_loss"]
    else:
        P = O.params_from(S.synth_state_dict(shapes, 0), O.TACORL_FROZEN)
        opt = O.new_tacorl_opt_state(P)

        def step(batch, s):
            torch.manual_seed(1000 + s)
            noise = O.draw_tacorl_noise(B, latent=wl["latent"])
            return O.tacorl_training_step(P, opt, batch, noise, cfg, 0)[0]["q1_loss"]
    return step


def time_reference_cpu(wl, B, steps, warmup, threads):
    from oracle import synth as S
    torch.set_num_threads(threads)
    kind = reference_kind()
    step = build_reference(wl, "cpu")[1] if kind == "reference" else port_step(wl, B)
    batch = reference_batch(wl, B)
    times = []
    for s in range(warmup + steps):
        torch.manual_seed(1000 + s)
        b = S.clone_batch(batch)          # a fresh dict per call: the reference mutates batch["states"] in place
        t0 = time.perf_counter()
        step(b, s)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
    return times, kind


def time_reference_gpu_eager(wl, B, steps=5, warmup=2):
    """The same reference modules on cuda:0 under torch eager: fp32 (cuDNN TF32 convolutions, torch's default) and bf16
    autocast.  Not the graded baseline; the honest bar (BASELINE.md section 3)."""
    from oracle import synth as S
    if not torch.cuda.is_available() or reference_kind() != "reference":
        return None
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    out = {}
    batch = reference_batch(wl, B)
    batch = to_device(batch, dev)
    for mode in ("fp32_tf32conv", "bf16_autocast"):
        try:
            m, step = build_reference(wl, dev)
            ac = torch.autocast("cuda", dtype=torch.bfloat16, enabled=(mode == "bf16_autocast"))
            for s in range(warmup):
                with ac:
                    step(S.clone_batch(batch), s)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for s in range(steps):
                with ac:
                    loss = step(S.clone_batch(batch), s)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[mode] = {"ms_per_step": ms, "value": B * frames_per_window(wl) / (ms / 1e3), "unit": "frames/s", "steps": steps,
                         "loss": float(loss.detach()) if torch.is_tensor(loss) else None}
            del m, step
            torch.cuda.empty_cache()
        except Exception as e:  # pragma: no cover - reported, not fatal
            out[mode] = {"error": repr(e)[:300]}
    out["note"] = ("unmodified reference modules, torch eager on cuda:0, batch resident on the device; step includes the "
                   "reference's per-step batch clone")
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    threads = os.cpu_count() or 1
    wl = WORKLOADS[args.workload]
    B = windows_per_gpu(args, world)

    def cpu_line(name, steps, warmup):
        w = WORKLOADS[name]
        times, kind = time_reference_cpu(w, B, steps, warmup, threads)
        ms = 1e3 * statistics.median(times)
        fps = B * frames_per_window(w) / (ms / 1e3)
        what = ("UNMODIFIED reference modules (oracle/_ref, vendored from /root/reference) + their own torch.optim.Adam"
                if kind == "reference" else "oracle port of the reference step (the vendored reference tree is absent)")
        return {"metric": w["metric"], "value": fps, "unit": "frames/s", "ms_per_step": ms,
                "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": kind, "ms_per_step": ms,
                                 "sample": f"median of {steps} timed steps (+{warmup} warm-up) of {B} windows x {frames_per_window(w)} frames: {what}, "
                                           f"torch CPU fp32, {threads} threads"},
                "workload": w["desc"]}

    main = cpu_line(args.workload, args.steps, args.warmup)
    line = {"impl": "reference", "metric": main["metric"], "value": main["value"], "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["desc"], "windows_per_step": B, "host": "cpu", "frames_per_window": frames_per_window(wl)},
            "cpu_baseline": main["cpu_baseline"],
            "e2e": {"value": main["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if args.workload == "play_lmp" and not args.no_tacorl:
        try:
            line["tacorl"] = cpu_line("tacorl", max(2, min(args.steps, 5)), 1)
        except Exception as e:  # pragma: no cover
            line["tacorl"] = {"error": repr(e)[:300]}
    if not args.no_gpu_eager:
        try:
            ge = time_reference_gpu_eager(wl, B)
            if ge is not None:
                line["reference_gpu_eager"] = ge
            if args.workload == "play_lmp" and not args.no_tacorl and ge is not None:
                line["tacorl"]["reference_gpu_eager"] = time_reference_gpu_eager(WORKLOADS["tacorl"], B)
        except Exception as e:  # pragma: no cover
            line["reference_gpu_eager"] = {"error": repr(e)[:300]}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------- our arm
def teardown(ctx):
    """Leave together.  Captured graphs reference the communicator's streams: release them before the group; if
    destroy_process_group() still does not return within a minute, say so and exit (everything is already printed)."""
    import gc
    import threading
    if ctx.world <= 1:
        return
    ctx.graphs.clear()
    gc.collect()
    ctx.barrier()
    from tacorl_b200 import parallel
    parallel.NativeAllReduce.shutdown()          # the library's own communicator (tacorl_dp_allreduce_*)
    done = threading.Event()

    def destroy():
        try:
            ctx.dist.destroy_process_group()
        finally:
            done.set()

    th = threading.Thread(target=destroy, daemon=True)
    th.start()
    th.join(timeout=60)
    sys.stdout.flush()
    if not done.is_set():
        sys.stderr.write(f"[bench rank {ctx.rank}] destroy_process_group() did not return within 60 s; exiting\n")
        sys.stderr.flush()
        os._exit(0)


def run_ours(args):
    ctx = Ctx(args)
    dist, world, rank, dev = ctx.dist, ctx.world, ctx.rank, ctx.dev
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line
        # the gradient all-reduce runs under the encoder backward: 16 NCCL channels on the 16 SMs the persistent
        # convolution kernels leave free (parallel.attach_data_parallel; scripts/n2_reserve_sweep.sh)
        from tacorl_b200.parallel import collective_channels
        os.environ.setdefault("NCCL_MAX_NCHANNELS", str(collective_channels(world)))
        os.environ.setdefault("NCCL_MIN_NCHANNELS", str(collective_channels(world)))
        # NCCL announces its version on stdout when the image sets NCCL_DEBUG: send its log to stderr, and route
        # fd 1 to stderr while the communicator comes up, so that stdout carries the JSON line and nothing else
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    trace("process group up")
    pk, pk_kind = peaks()
    B = windows_per_gpu(args, world)
    wl = WORKLOADS[args.workload]

    main, h = measure_workload(ctx, args.workload, args.precision, args.steps, args.warmup, sample_clocks=True,
                               dump_dir=args.dump_outputs)
    rooflines = []
    if "rgb_static" in wl["mods"] and args.precision == "bf16" and wl["module"] != "cql":
        try:
            if wl["module"] == "play_lmp":
                rooflines.append(roofline_encoder(ctx, h, main["ms_per_step"], pk, pk_kind))
            rooflines.append(roofline_recurrence(ctx, h, main["ms_per_step"], pk, pk_kind))
            if wl["module"] == "play_lmp":
                rooflines.append(roofline_adam(ctx, h, pk, pk_kind))
        except Exception as e:  # pragma: no cover - reported, never fatal for the headline metric
            sys.stderr.write(f"[bench] roofline probe failed: {e!r}\n")
    del h
    ctx.graphs.clear()
    torch.cuda.empty_cache()

    extra = {}
    if args.workload == "play_lmp" and not args.no_tacorl:
        try:
            tac, th = measure_workload(ctx, "tacorl", args.precision, args.steps, args.warmup)
            tac["q1_loss"] = tac.pop("final_loss", None)
            extra["tacorl"] = tac
            del th
            ctx.graphs.clear()
            torch.cuda.empty_cache()
        except Exception as e:  # pragma: no cover
            sys.stderr.write(f"[bench] TACO-RL measurement failed: {e!r}\n")
            extra["tacorl"] = {"error": repr(e)[:300]}
    if args.workload == "play_lmp" and args.precision == "bf16" and not args.no_fp32 and world == 1:
        # BASELINE configs[1] asks for fp32 and bf16: the fp32 SIMT parity path, short run, resident inputs only
        try:
            f32, fh = measure_workload(ctx, "play_lmp", "fp32", max(3, min(10, args.steps)), 3, e2e=False)
            extra["fp32"] = {k: f32[k] for k in ("value", "unit", "ms_per_step", "launches_per_step", "cuda_graph")}
            extra["fp32"]["note"] = "same workload on the fp32 FFMA parity path (ops.set_precision('fp32')), resident inputs"
            del fh
            ctx.graphs.clear()
            torch.cuda.empty_cache()
            from tacorl_b200 import ops
            ops.set_precision(args.precision)
        except Exception as e:  # pragma: no cover
            extra["fp32"] = {"error": repr(e)[:300]}

    if rank == 0:
        line = {
            "metric": main["metric"], "value": main["value"], "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
            "config": {"workload": wl["desc"], "windows_per_gpu": B, "global_windows": B * world,
                       "frames_per_window": frames_per_window(wl), "parallelism": f"dp{world}", "precision": args.precision,
                       "cuda_graph": main["cuda_graph"],
                       "input": "uint8 frames, ScaleImageTensor+Normalize fused into the first kernel" if args.input == "u8"
                                else "float32 frames (pre-normalised on the host)",
                       "l2_policy": f"inputs ({main['e2e']['h2d_bytes_per_step'] / 1e6:.0f} MB/step) + activations "
                                    "(> 1 GB/step) exceed the 126 MB L2"},
            "e2e": main["e2e"], "gpu_launches": main["gpu_launches"], "launches_per_step": main["launches_per_step"],
            "clocks": main.get("clocks"),
            "roofline": rooflines[0] if rooflines else None,
            "rooflines": rooflines,
            "algorithmic_tflops_whole_step": main["algorithmic_tflops_whole_step"],
            "final_loss": main.get("final_loss"),
        }
        line.update(extra)
        if not args.no_cpu_baseline and world == 1:
            threads = os.cpu_count() or 1
            try:
                t, kind = time_reference_cpu(wl, B, args.cpu_steps, 1, threads)
                cms = 1e3 * statistics.median(t)
                line["cpu_baseline"] = {"value": B * frames_per_window(wl) / (cms / 1e3), "unit": "frames/s", "cores": threads,
                                        "kind": kind, "ms_per_step": cms,
                                        "sample": f"median of {args.cpu_steps} timed steps (+1 warm-up) of the same {B} windows x "
                                                  f"{frames_per_window(wl)} frames workload: " + ("unmodified reference modules (oracle/_ref)"
                                                  if kind == "reference" else "oracle port of the reference step") +
                                                  f", torch CPU fp32, {threads} threads"}
            except Exception as e:  # pragma: no cover
                line["cpu_baseline"] = {"error": repr(e)[:300]}
        print(json.dumps(line), flush=True)
    teardown(ctx)


def main():
    args = parse()
    if os.environ.get("BENCH_TRACE"):       # where is each rank when a wrapper's timeout sends SIGTERM?
        import faulthandler
        import signal
        faulthandler.register(signal.SIGTERM, all_threads=False, chain=True)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
