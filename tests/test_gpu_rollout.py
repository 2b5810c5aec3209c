"""GPU tests of the batched rollout policy (tacorl_b200/rollout.py, csrc/rollout.cu, DESIGN.md section 16): the decoder
step teacher-forced stage by stage against fp64, batch invariance, the whole policy against the CPU oracle, graph
replays against eager runs, and the policy's use of the module's weights."""
import numpy as np
import pytest
import torch

from oracle import replay_oracle as RO
from oracle import rollout_oracle as R
from oracle import synth as S
from oracle import tacorl_oracle as O
from tests import rnn_bf16_oracle as RB
from tests.gpu_util import DEV, assert_close, build_play_lmp, build_tacorl, double_params, parity_report

pytestmark = pytest.mark.gpu

TAU = RB.TAU      # per-element bar |got - want| <= TAU * scale, both precisions (fp32 accumulation of <= 4096 terms)
CONTROLS = ("restart_ignored", "u1_u2_swapped", "draw_off_by_one", "stale_layer0")


def _decoder(P, E, H, seed=4):
    from tacorl_b200.networks.action_decoders.action_decoder_logistic import ActionDecoderLogistic
    torch.manual_seed(seed)
    d = ActionDecoderLogistic(state_dim=E, latent_plan_dim=P, hidden_size=H)
    with torch.no_grad():     # heads at a scale where the mixture logits spread
        for fc in (d.prob_fc, d.mean_fc, d.log_scale_fc, d.gripper_fc):
            fc.weight.mul_(4.0)
    return d.to(DEV).eval()


def _uniforms_shifted(seed, t, env, shift=0, swap=False):
    """The oracle's uniforms, or a control: draw index shifted by `shift`, or u1 / u2 taken from the wrong uniforms."""
    u = []
    for tt, e in zip(t, env):
        words = RO.philox4x32_10(int(tt) & 0xFFFFFFFF, int(tt) >> 32, int(e), np.arange(17) + shift, seed & 0xFFFFFFFF,
                                 seed >> 32)
        w = np.stack(words, -1).reshape(-1)[:66]           # uniform i = word i % 4 of draw i // 4
        u.append((w >> 8).astype(np.float32) * np.float32(2.0 ** -24))
    u = torch.from_numpy(np.stack(u))
    if swap:
        return u[:, 6:].reshape(-1, 6, 10), u[:, :6]
    return u[:, :60].reshape(-1, 6, 10), u[:, 60:]


def _step_inputs(n, P, E, H, seed):
    g = torch.Generator().manual_seed(seed)
    plan = torch.tanh(torch.randn(n, P, generator=g))
    emb = torch.randn(n, E, generator=g)
    hidden = torch.relu(torch.randn(2, n, H, generator=g)) * 0.5
    restart = (torch.arange(n) % 3 == 1).int()           # rows 1, 4, 7, ... start over
    env = torch.randint(0, 1000, (n,), generator=g, dtype=torch.int32)
    t = torch.randint(0, 1 << 40, (n,), generator=g, dtype=torch.int64)
    return plan, emb, hidden, restart, env, t


def _run_step(dec, plan, emb, hidden, restart, env, t, seed):
    from tacorl_b200.rollout import decoder_step
    n = plan.shape[0]
    d = {k: v.to(DEV).contiguous() for k, v in dict(plan=plan, emb=emb, hidden=hidden, restart=restart, env=env, t=t).items()}
    acts = torch.empty(n, 7, device=DEV)
    logits = torch.empty(n, 182, device=DEV)
    decoder_step(dec, d["plan"], d["emb"], d["hidden"], d["restart"], seed, d["env"], d["t"], acts, logits)
    torch.cuda.synchronize()
    return d["hidden"].cpu(), logits.cpu(), acts.cpu(), d["t"].cpu()


def _fp32_fwd(x, w_ih, w_hh, b_ih, b_hh, h0):
    x, w_ih, w_hh, h0 = x.double(), w_ih.double(), w_hh.double(), h0.double()
    b = b_ih.double() + b_hh.double()
    return torch.relu(x @ w_ih.t() + b + h0 @ w_hh.t()), x.abs() @ w_ih.abs().t() + b.abs() + h0.abs() @ w_hh.abs().t()


def _check_step(dec, inputs, got, precision, seed, control=None):
    """Every stage of one kernel step against fp64 on the kernel's own inputs.  Returns {stage: (ok, worst ratio)}."""
    plan, emb, h_prev, restart, env, t = inputs
    hid, logits, acts, t_after = got
    from tacorl_b200.rollout import decoder_weights
    w = [x.cpu() for x in decoder_weights(dec)]
    keep = (restart == 0).double().view(1, -1, 1) if control != "restart_ignored" else torch.ones(1, plan.shape[0], 1)
    h0 = h_prev.double() * keep
    x0 = torch.cat([plan, emb], 1)
    x1 = hid[0] if control != "stale_layer0" else h0[0]
    res = {}
    for l, x in ((0, x0), (1, x1)):
        wi, wh, bi, bh = w[4 * l:4 * l + 4]
        if precision == "bf16":
            want, scale = RB.fwd(x[None], wi, wh, bi, bh, hid[l][None], h0=h0[l])["out"]
            want, scale = want[0], scale[0]
        else:
            want, scale = _fp32_fwd(x, wi, wh, bi, bh, h0[l])
        ok, ratio = RB.check(hid[l], want, scale, TAU)[:2]
        res[f"layer{l}"] = (ok, ratio)
    W = torch.cat(w[8::2], 0).double()
    b = torch.cat(w[9::2], 0).double()
    h1 = RB.rne(hid[1]) if precision == "bf16" else hid[1].double()
    Wr = RB.rne(W) if precision == "bf16" else W
    ok, ratio = RB.check(logits, h1 @ Wr.t() + b, h1.abs() @ Wr.abs().t() + b.abs(), TAU)[:2]
    res["logits"] = (ok, ratio)
    shift = 1 if control == "draw_off_by_one" else 0
    u1, u2 = _uniforms_shifted(seed, t.tolist(), env.tolist(), shift, control == "u1_u2_swapped")
    lg = logits.double()
    lp, mm, ls, grip = lg[:, :60].view(-1, 1, 6, 10), lg[:, 60:120].view(-1, 1, 6, 10), lg[:, 120:180], lg[:, 180:]
    ls = torch.clamp(ls, min=-5.0).view(-1, 1, 6, 10)
    want = O.dlm_sample(lp, ls, mm, grip.view(-1, 1, 2), u1.double()[:, None], u2.double()[:, None])[:, 0]
    # the mixture pick may differ only where the top two Gumbel scores are within 1e-5
    r1, r2 = 1e-5, 1.0 - 1e-5
    score = lp[:, 0] - torch.log(-torch.log((r1 - r2) * u1.double() + r2))
    top2 = score.topk(2, dim=-1).values
    near_tie = (top2[..., 0] - top2[..., 1]) < 1e-5
    close = (acts[:, :6].double() - want[:, :6]).abs() <= 1e-4 * (1.0 + want[:, :6].abs())
    ok = bool((close | near_tie).all()) and torch.equal(acts[:, 6].double(), want[:, 6])
    res["actions"] = (ok, float((acts.double() - want).abs().max()))
    res["t"] = (torch.equal(t_after, t + 1), 0.0)
    return res


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("P,E", [(16, 32), (32, 64)])
@pytest.mark.parametrize("H", [64, 2048])
@pytest.mark.parametrize("n", [1, 5, 64])
def test_decoder_step_teacher_forced(n, H, P, E, precision):
    from tacorl_b200 import ops
    ops.set_precision(precision)
    try:
        dec = _decoder(P, E, H)
        seed = 0xC0FFEE12345
        inputs = _step_inputs(n, P, E, H, seed=n * 7 + H)
        got = _run_step(dec, *inputs, seed)
        res = _check_step(dec, inputs, got, precision, seed)
        parity_report(f"rollout_step_{precision}_n{n}_H{H}_I{P + E}", {k: list(v) for k, v in res.items()})
        assert all(ok for ok, _ in res.values()), res
        # the kernel's action equals the library's dlm_sample on its logits and the same uniforms, bit for bit
        u1, u2 = R.uniforms(seed, inputs[5].numpy(), inputs[4].numpy())
        pred, _ = ops.dlm_sample(got[1].to(DEV), u1.reshape(n, 60).to(DEV), u2.to(DEV), None,
                                 *dec._grip)
        assert torch.equal(pred.cpu(), got[2])
        # the controls must fail (a restart flag only matters on a row with a non-zero previous state)
        for control in CONTROLS:
            if control == "restart_ignored" and n < 2:
                continue
            bad = _check_step(dec, inputs, got, precision, seed, control)
            assert not all(ok for ok, _ in bad.values()), (control, bad)
    finally:
        ops.set_precision("fp32")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_batch_invariance(precision):
    """Every row of a 64-environment step is bit-identical to the same row stepped alone."""
    from tacorl_b200 import ops
    ops.set_precision(precision)
    try:
        dec = _decoder(16, 32, 2048)
        inputs = _step_inputs(64, 16, 32, 2048, seed=5)
        hid, logits, acts, t = _run_step(dec, *inputs, 77)
        for r in (0, 1, 2, 7, 31, 32, 63):
            plan, emb, h, rs, env, tt = inputs
            one = _run_step(dec, plan[r:r + 1], emb[r:r + 1], h[:, r:r + 1], rs[r:r + 1], env[r:r + 1], tt[r:r + 1], 77)
            assert torch.equal(one[0], hid[:, r:r + 1]), r
            assert torch.equal(one[1], logits[r:r + 1]), r
            assert torch.equal(one[2], acts[r:r + 1]), r
            assert torch.equal(one[3], t[r:r + 1]), r
        # and a batch of 5 agrees with the same rows of the batch of 64 (row tiles of different sizes)
        five = _run_step(dec, *[x[:5] if x.dim() < 3 else x[:, :5] for x in inputs], 77)
        assert torch.equal(five[2], acts[:5]) and torch.equal(five[0], hid[:, :5])
    finally:
        ops.set_precision("fp32")


# ------------------------------------------------------------------------------------------------ whole policy
def _tacorl(hidden, mods=("rgb_static",), latent=16, seed=21, precision="fp32"):
    lmp = build_play_lmp("tanh_net", mods, hidden, latent, 8, goal_modalities=mods)
    t = build_tacorl(lmp, precision)
    shapes = {k: list(v.shape) for k, v in t.state_dict().items()}
    sd = S.synth_state_dict(shapes, seed)
    t.load_state_dict(sd, strict=True)
    return t.to(DEV).eval(), sd


def _sizes(mods):
    return {"rgb_static": 200, "rgb_gripper": 84}


def _schedule(n, steps):
    """Staggered episode events: {step: [(kind, rows)]}; every row replans at most every 6 steps."""
    ev = {0: [("reset", list(range(n)))]}
    for s in range(1, steps):
        e = []
        for r in range(n):
            k = (s + 2 * r) % 6
            if k == 0 and s % 12 == 0:
                e.append(("reset", [r]))
            elif k == 0 and (s + r) % 3 == 0:
                e.append(("set_goal", [r]))
            elif k == 0:
                e.append(("replan", [r]))
        if e:
            ev[s] = e
    return ev


def _drive(policy, oracle, mods, n, steps, seed, gold=None):
    """Run policy (and the oracle) through the schedule; returns per-step actions (and the oracle's)."""
    sz = _sizes(mods)
    got, want = [], []
    for s in range(steps):
        for kind, rows in _schedule(n, steps).get(s, []):
            if kind == "replan":
                policy.replan(rows)
                if oracle:
                    oracle.replan(rows)
                continue
            goal = {m: S.synth_images((len(rows), 3, sz[m], sz[m]), seed, f"goal{s}_{rows[0]}_{m}") for m in mods}
            getattr(policy, kind)(rows, {m: v.to(DEV) for m, v in goal.items()})
            if oracle:
                getattr(oracle, kind)(rows, goal)
        obs = {m: S.synth_images((n, 3, sz[m], sz[m]), seed, f"obs{s}_{m}") for m in mods}
        got.append(policy.step({m: v.to(DEV) for m, v in obs.items()}).cpu().clone())
        if oracle:
            want.append(oracle.step(obs)[0].float())
    return torch.stack(got), (torch.stack(want) if oracle else None)


@pytest.mark.parametrize("precision,mods,hidden,n,steps", [
    ("fp32", ("rgb_static",), 2048, 8, 24),
    ("bf16", ("rgb_static",), 2048, 8, 24),
    ("fp32", ("rgb_static", "rgb_gripper"), 2048, 4, 12),
])
def test_policy_matches_oracle(precision, mods, hidden, n, steps):
    from tacorl_b200 import ops
    from tacorl_b200.rollout import RolloutPolicy
    latent = 32 if len(mods) > 1 else 16
    t, sd = _tacorl(hidden, mods, latent, precision=precision)
    try:
        ops.set_precision(precision)
        policy = RolloutPolicy(t, n, seed=1234, env_ids=[100 + 3 * r for r in range(n)])
        oracle = R.RolloutOracle(double_params(sd), n, hidden, latent, seed=1234, env_ids=[100 + 3 * r for r in range(n)],
                                 obs_mods=mods, goal_mods=mods)
        got, want = _drive(policy, oracle, mods, n, steps, seed=6)
        if precision == "fp32":
            assert_close("rollout actions", got, want, 1e-4, atol=1e-5)
        else:   # the criterion of test_rollout_inner_loop_matches_oracle: gripper + most dims agree
            assert torch.equal(got[..., -1], want[..., -1])
            close = ((got[..., :6] - want[..., :6]).abs() < 5e-2).float().mean()
            assert close > 0.8, close
        parity_report(f"rollout_policy_{precision}_{len(mods)}view",
                      {"max_abs": float((got - want).abs().max()), "launches": {str(k): v for k, v in policy.launches.items()}})
    finally:
        ops.set_precision("fp32")


@pytest.mark.parametrize("precision,mods", [("fp32", ("rgb_static",)), ("bf16", ("rgb_static",)),
                                            ("bf16", ("rgb_static", "rgb_gripper"))])
def test_graph_replays_equal_eager_runs(precision, mods):
    from tacorl_b200 import ops
    from tacorl_b200.rollout import RolloutPolicy
    t, _ = _tacorl(2048, mods, 32 if len(mods) > 1 else 16, precision=precision)
    try:
        ops.set_precision(precision)
        a, _ = _drive(RolloutPolicy(t, 6, seed=9), None, mods, 6, 14, seed=2)
        b, _ = _drive(RolloutPolicy(t, 6, seed=9, use_graphs=False), None, mods, 6, 14, seed=2)
        assert torch.equal(a, b)
    finally:
        ops.set_precision("fp32")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_module_weights_and_live_parameters(precision):
    from tacorl_b200 import _lib, ops
    from tacorl_b200.rollout import RolloutPolicy, decoder_step
    t, _ = _tacorl(256, precision=precision)
    try:
        ops.set_precision(precision)
        opts = t.configure_optimizers()     # the decoder's bf16 shadows exist, as after training
        w = t.action_decoder.rnn.weight_hh_l1
        assert (ops.shadow_of(w) is not None) == (precision == "bf16")
        before = {k: v.clone() for k, v in t.state_dict().items()}
        p1, p2 = RolloutPolicy(t, 3, seed=5), RolloutPolicy(t, 3, seed=5)
        mods = ("rgb_static",)
        _drive(p1, None, mods, 3, 4, seed=3)
        _drive(p2, None, mods, 3, 4, seed=3)
        for k, v in t.state_dict().items():
            assert torch.equal(v, before[k]), k
        assert all(p.grad is None for p in t.parameters())
        # a torch-side edit of a decoder weight between steps reaches the next step (graph replay)
        obs = {"rgb_static": S.synth_images((3, 3, 200, 200), 3, "edit").to(DEV)}
        with torch.no_grad():
            w.mul_(1.5)
        edited = p1.step(obs).clone()
        with torch.no_grad():
            w.copy_(before["action_decoder.rnn.weight_hh_l1"])
        orig = p2.step(obs).clone()
        assert not torch.equal(edited, orig)
        # the decoder step is 3 library launches
        n0 = _lib.launch_count()
        decoder_step(t.action_decoder, p1.plan, torch.zeros(3, 32, device=DEV), p1.hidden, p1.restart, 0, p1.env_id,
                     p1.t, p1.actions)
        assert _lib.launch_count() - n0 == 3
        assert len(opts) > 0
    finally:
        ops.set_precision("fp32")


# library launches per replayed step and per replan step, as DESIGN.md section 16 states them
DESIGN_LAUNCHES = [("bf16", ("rgb_static",), 10, 19), ("fp32", ("rgb_static",), 13, 25),
                   ("bf16", ("rgb_static", "rgb_gripper"), 17, 33)]


@pytest.mark.parametrize("precision,mods,step,replan_step", DESIGN_LAUNCHES)
def test_launches_per_step_are_the_documented_ones(precision, mods, step, replan_step):
    from tacorl_b200 import ops
    from tacorl_b200.rollout import RolloutPolicy
    t, _ = _tacorl(256, mods, 32 if len(mods) > 1 else 16, precision=precision)
    try:
        ops.set_precision(precision)
        p = RolloutPolicy(t, 4, seed=1)
        _drive(p, None, mods, 4, 3, seed=4)          # a replan step, then plain steps
        assert p.launches == {(True, precision): replan_step, (False, precision): step}
        parity_report(f"rollout_launches_{precision}_{len(mods)}view", {"step": step, "replan_step": replan_step})
    finally:
        ops.set_precision("fp32")


def _both(pg, pe, obs):
    return pg.step(obs).cpu().clone(), pe.step(obs).cpu().clone()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_optimiser_built_after_capture_is_seen(precision):
    """An optimiser created after the graphs were captured moves the parameters into its flat buffer: the policy
    recaptures, and a later torch edit reaches the replayed step exactly as it reaches an eager one."""
    from tacorl_b200 import ops
    from tacorl_b200.rollout import RolloutPolicy
    t, _ = _tacorl(256, precision=precision)
    try:
        ops.set_precision(precision)
        mods = ("rgb_static",)
        pg, pe = RolloutPolicy(t, 3, seed=8), RolloutPolicy(t, 3, seed=8, use_graphs=False)
        a, b = _drive(pg, None, mods, 3, 4, seed=5)[0], _drive(pe, None, mods, 3, 4, seed=5)[0]
        assert torch.equal(a, b)
        captures = pg.captures
        w = t.action_decoder.rnn.weight_hh_l1
        old_ptr = w.data_ptr()
        opts = t.configure_optimizers()
        assert w.data_ptr() != old_ptr           # the parameters now live in the optimiser's flat buffer
        obs = {"rgb_static": S.synth_images((3, 3, 200, 200), 5, "after").to(DEV)}
        g, e = _both(pg, pe, obs)
        assert torch.equal(g, e) and pg.captures > captures
        with torch.no_grad():
            w.mul_(1.5)
        g2, e2 = _both(pg, pe, obs)
        assert torch.equal(g2, e2) and not torch.equal(g2, g)
        assert len(opts) > 0
    finally:
        ops.set_precision("fp32")


def test_dropped_optimiser_shadows_are_not_read():
    """bf16: graphs captured while an optimiser's bf16 shadows exist stay correct after the optimiser is dropped."""
    import gc
    from tacorl_b200 import ops
    from tacorl_b200.rollout import RolloutPolicy
    t, _ = _tacorl(256, precision="bf16")
    try:
        ops.set_precision("bf16")
        mods = ("rgb_static",)
        opts = t.configure_optimizers()
        w = t.action_decoder.rnn.weight_hh_l1
        assert ops.shadow_of(w) is not None
        pg, pe = RolloutPolicy(t, 3, seed=8), RolloutPolicy(t, 3, seed=8, use_graphs=False)
        a, b = _drive(pg, None, mods, 3, 4, seed=5)[0], _drive(pe, None, mods, 3, 4, seed=5)[0]
        assert torch.equal(a, b)
        obs = {"rgb_static": S.synth_images((3, 3, 200, 200), 5, "drop").to(DEV)}
        with torch.no_grad():
            w.mul_(1.5)
        g, e = _both(pg, pe, obs)
        assert torch.equal(g, e)
        captures = pg.captures
        del opts
        gc.collect()
        assert ops.shadow_of(w) is None
        with torch.no_grad():
            w.mul_(0.5)
        g2, e2 = _both(pg, pe, obs)
        assert torch.equal(g2, e2) and not torch.equal(g2, g) and pg.captures > captures
    finally:
        ops.set_precision("fp32")


def test_policy_rejects_mismatched_inputs():
    from tacorl_b200.rollout import RolloutPolicy
    t, _ = _tacorl(64)
    p = RolloutPolicy(t, 2)
    img = torch.zeros(2, 3, 84, 84, dtype=torch.uint8, device=DEV)
    with pytest.raises(ValueError, match="no goal"):
        p.step({"rgb_static": img})
    with pytest.raises(ValueError, match="out of range"):
        p.reset([2], {"rgb_static": img[:1]})
    with pytest.raises(ValueError, match="modalities"):
        p.reset([0, 1], {"rgb_gripper": img})
    p.reset([0, 1], {"rgb_static": img})
    p.step({"rgb_static": img})
    with pytest.raises(ValueError, match="static buffer"):
        p.step({"rgb_static": torch.zeros(2, 3, 96, 96, dtype=torch.uint8, device=DEV)})
    with pytest.raises(ValueError, match="static buffer"):
        p.step({"rgb_static": img.float()})
