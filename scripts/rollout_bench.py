#!/usr/bin/env python
"""Batched rollout policy (tacorl_b200.rollout.RolloutPolicy) on one GPU, bf16, against today's eager loop.

    python scripts/rollout_bench.py --out DIR [--steps 1000] [--warmup 50] [--agents single_view,multi_view]

For n_envs in {1, 8, 64} and the single-view (static 200x200, latent 16) and multi-view (static 200x200 + gripper
84x84, latent 32) TACO-RL agents, hidden 2048, writes DIR/rollout_bench.json with:
  graphed_step_ms     one policy step (one CUDA-graph replay, no replan), CUDA events over --steps steps;
  replan_step_ms      the same with every row replanning (the replan graph);
  eager_loop_ms       the reference's per-step calls at the same batch: perceptual_encoder.get_state_from_observation +
                      action_decoder.act() (one shared hidden state, torch.rand noise);
  decoder_step        tacorl_rollout_decoder_step alone: us per call back to back (its weights then come from L2, they fit
                      in the 126 MB) and after overwriting a 512 MB buffer before each call (weights from HBM), the
                      weight bytes it reads and those bytes over each time;
  launches            library launches per replayed step and per replan step;
  device              name and power limit of the GPU, read in the same run.
--agents play_lmp,play_lmp_sampled,cql_flat,cql_flat_sampled,tacorl_sampled (single-view, static 200x200) writes
DIR/rollout_baselines_bench.json instead, with per agent and n_envs: graphed_step_ms, replan_step_ms (agents with a
plan), eager_loop_ms (the reference's per-step calls: encoder + act() for PlayLMP and TACO-RL, the actor's
get_actions(deterministic=True) on the encoder and cached goal embeddings for flat CQL), sampler_us
(tacorl_rollout_policy_sample alone, CUDA events over back-to-back calls, on the plan for PlayLMP / TACO-RL and on the
actions + gripper for flat CQL), launches and device.
Weights and inputs are synthetic (seeded)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

AGENTS = {"single_view": (("rgb_static",), 16), "multi_view": (("rgb_static", "rgb_gripper"), 32)}
BASELINES = {"play_lmp": True, "play_lmp_sampled": False, "cql_flat": True, "cql_flat_sampled": False,
             "tacorl_sampled": False}           # agent -> deterministic
SIZE = {"rgb_static": 200, "rgb_gripper": 84}


def device_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        info["power_limit_and_max_sm_clock"] = subprocess.run(
            ["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
            capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # pragma: no cover
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e!r}"
    return info


def build(mods, latent, hidden):
    from oracle import synth as S
    from tests.gpu_util import build_play_lmp, build_tacorl
    lmp = build_play_lmp("tanh_net", mods, hidden, latent, 16, goal_modalities=mods)
    m = build_tacorl(lmp, "bf16")
    sd = S.synth_state_dict({k: list(v.shape) for k, v in m.state_dict().items()}, 3)
    m.load_state_dict(sd)
    return m.cuda().eval()


def build_baseline(agent, hidden):
    from oracle import synth as S
    from tests.gpu_util import build_cql_flat, build_play_lmp, build_tacorl
    mods = ("rgb_static",)
    if agent.startswith("play_lmp"):
        m = build_play_lmp("tanh_net", mods, hidden, 16, 16, goal_modalities=mods)
    elif agent.startswith("cql"):
        m = build_cql_flat("bf16")
    else:
        m = build_tacorl(build_play_lmp("tanh_net", mods, hidden, 16, 16, goal_modalities=mods), "bf16")
    m.load_state_dict(S.synth_state_dict({k: list(v.shape) for k, v in m.state_dict().items()}, 3))
    return m.cuda().eval()


def run_baseline(agent, m, n, args):
    from oracle import synth as S
    from tacorl_b200.rollout import RolloutPolicy, policy_sample
    obs = {"rgb_static": S.synth_images((n, 3, 200, 200), 1, "orgb_static").mul(127.5).add(127.5).round()
           .to(torch.uint8).cuda()}
    pol = RolloutPolicy(m, n, seed=0, deterministic=BASELINES[agent])
    pol.reset(list(range(n)), obs)
    pol.step(obs)
    row = {"agent": agent, "n_envs": n, "graphed_step_ms": timed(lambda: pol.step(), args.steps, args.warmup)}
    if pol.kind != "cql":
        def replan_step():
            pol.replan(list(range(n)))
            pol.step()
        row["replan_step_ms"] = timed(replan_step, args.steps, args.warmup)

        def eager():
            with torch.no_grad():
                s = m.perceptual_encoder.get_state_from_observation(observation=obs, modalities=m.action_decoder_modalities)
                m.action_decoder.act(latent_plan=pol.plan, perceptual_emb=s.reshape(n, 1, -1))
        m.action_decoder.clear_hidden_state()
        row["eager_loop_ms"] = timed(eager, max(100, args.steps // 10), 10)
        m.action_decoder.clear_hidden_state()
        A, logits, mask, out = pol.P, None, pol.restart, pol.plan
    else:
        actor = m.actor

        def eager():
            with torch.no_grad():
                e = actor.encoder.get_state_from_observation(observation=obs, modalities=actor.env_modalities)
                actor.actor.get_actions(torch.cat([e.reshape(n, -1), pol.goal_emb], -1), deterministic=True)
        row["eager_loop_ms"] = timed(eager, max(100, args.steps // 10), 10)
        A, logits, mask, out = 6, torch.zeros(n, 2, device="cuda"), None, pol.actions
    mean, std = torch.zeros(n, A, device="cuda"), torch.ones(n, A, device="cuda")
    t = torch.zeros(n, device="cuda", dtype=torch.int64)
    row["sampler_us"] = 1e3 * timed(lambda: policy_sample(mean, std, logits, mask, 0, pol.env_id, t, out, True),
                                    args.steps, args.warmup)
    row["launches"] = {str(k): v for k, v in pol.launches.items()}
    return row


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def timed_cold(fn, steps, warmup, flush):
    """Mean time of fn with the L2 overwritten (a 512 MB fill) before each call, events around fn only."""
    for _ in range(warmup):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        flush.fill_(1.0)
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in ev) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--hidden", type=int, default=2048)
    ap.add_argument("--agents", default="single_view,multi_view",
                    help=f"comma-separated, from {sorted(AGENTS)} or from {sorted(BASELINES)}")
    args = ap.parse_args()
    agents = args.agents.split(",")
    unknown = [a for a in agents if a not in AGENTS and a not in BASELINES]
    if unknown or (any(a in AGENTS for a in agents) and any(a in BASELINES for a in agents)):
        raise SystemExit(f"--agents: {unknown or 'mixes the TACO-RL agents with the baselines'}")
    if not torch.cuda.is_available():
        raise SystemExit("rollout_bench needs a CUDA device")
    from oracle import synth as S
    from tacorl_b200 import ops
    from tacorl_b200.rollout import RolloutPolicy, decoder_step, decoder_weights
    ops.set_precision("bf16")
    res = {"device": device_info(), "precision": "bf16", "hidden": args.hidden, "steps": args.steps, "runs": []}
    if agents[0] in BASELINES:
        for agent in agents:
            m = build_baseline(agent, args.hidden)
            for n in (1, 8, 64):
                row = run_baseline(agent, m, n, args)
                res["runs"].append(row)
                print(json.dumps(row), flush=True)
            del m
            torch.cuda.empty_cache()
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "rollout_baselines_bench.json"), "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(res["device"]))
        return
    flush = torch.empty(128 << 20, device="cuda")
    for agent in agents:
        mods, latent = AGENTS[agent]
        m = build(mods, latent, args.hidden)
        for n in (1, 8, 64):
            obs = {k: S.synth_images((n, 3, SIZE[k], SIZE[k]), 1, f"o{k}").mul(127.5).add(127.5).round().to(torch.uint8).cuda()
                   for k in mods}
            pol = RolloutPolicy(m, n, seed=0)
            pol.reset(list(range(n)), obs)
            pol.step(obs)
            step_ms = timed(lambda: pol.step(), args.steps, args.warmup)

            def replan_step():
                pol.replan(list(range(n)))
                pol.step()
            replan_ms = timed(replan_step, args.steps, args.warmup)

            def eager():
                with torch.no_grad():
                    s = m.perceptual_encoder.get_state_from_observation(observation=obs, modalities=m.action_decoder_modalities)
                    m.action_decoder.act(latent_plan=pol.plan, perceptual_emb=s.reshape(n, 1, -1))
            m.action_decoder.clear_hidden_state()
            eager_ms = timed(eager, max(100, args.steps // 10), 10)
            m.action_decoder.clear_hidden_state()
            emb = torch.zeros(n, pol.E, device="cuda")

            def dec():
                decoder_step(m.action_decoder, pol.plan, emb, pol.hidden, pol.restart, 0, pol.env_id, pol.t, pol.actions,
                             None, pol.ws)
            dec_warm_ms = timed(dec, args.steps, args.warmup)
            dec_cold_ms = timed_cold(dec, min(args.steps, 300), 5, flush)
            ws = decoder_weights(m.action_decoder)
            wbytes = sum(w.numel() * (2 if ops.shadow_of(w) is not None else 4) for w in ws)
            row = {"agent": agent, "n_envs": n, "graphed_step_ms": step_ms, "replan_step_ms": replan_ms,
                   "eager_loop_ms": eager_ms,
                   "decoder_step": {"weight_bytes": wbytes, "weights_read_as": "bf16 copies" if wbytes < 3 * sum(w.numel() for w in ws) else "fp32",
                                    "us_back_to_back_weights_from_L2": dec_warm_ms * 1e3,
                                    "us_after_L2_overwrite_weights_from_HBM": dec_cold_ms * 1e3,
                                    "GBps_L2": wbytes / (dec_warm_ms * 1e-3) / 1e9,
                                    "GBps_HBM": wbytes / (dec_cold_ms * 1e-3) / 1e9},
                   "launches": {str(k): v for k, v in pol.launches.items()}}
            res["runs"].append(row)
            print(json.dumps(row), flush=True)
        del m
        torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "rollout_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["device"]))


if __name__ == "__main__":
    main()
