"""GPU tests of the rollout policy's sampler (tacorl_rollout_policy_sample) and of RolloutPolicy on PlayLMP and flat CQL,
deterministic and sampled, and on TACO-RL sampled (tacorl_b200/rollout.py, csrc/rollout.cu, DESIGN.md section 16): the
sampler against fp64 with controls that must fail, its batch invariance and distribution, the whole policy against the
CPU oracle, graph replays against eager runs, launch counts, and recapture after an optimiser is built."""
import numpy as np
import pytest
import torch

from oracle import replay_oracle as RO
from oracle import rollout_oracle as R
from oracle import synth as S
from tests import rollout_baselines_oracle as RB
from tests.gpu_util import DEV, assert_close, build_cql_flat, build_play_lmp, double_params, parity_report
from tests.test_gpu_rollout import _schedule, _sizes, _tacorl

pytestmark = pytest.mark.gpu

CONTROLS = ("ua_ub_swapped", "draws_from_0", "mask_ignored", "t_after_increment")
SENTINEL = 7.0


# ------------------------------------------------------------------------------------------------ the sampler
def _uniforms(seed, t, env, A, gripper, draw0=RB.POLICY_DRAW0, swap=False):
    """policy_uniforms, or a control: draws from `draw0`, or u_a / u_b swapped."""
    if draw0 == RB.POLICY_DRAW0:
        ua, ub, ug = RB.policy_uniforms(seed, t, env, A, gripper)
    else:
        w0, w1, _, _ = RO.philox4x32_10((t & 0xFFFFFFFF)[:, None], (t >> 32)[:, None], env[:, None],
                                        np.arange(draw0, draw0 + A + 1, dtype=np.uint64), seed & 0xFFFFFFFF, seed >> 32)
        ua, ub = RB._u24(w0), RB._u24(w1)
        ug = torch.stack([ua[:, A], ub[:, A]], -1) if gripper else None
        ua, ub = ua[:, :A], ub[:, :A]
    if swap:
        ua, ub = ub, ua
        ug = ug.flip(-1) if ug is not None else None
    return ua, ub, ug


def _sampler_inputs(n, A, seed):
    g = torch.Generator().manual_seed(seed)
    mean = torch.clamp(2.0 * torch.randn(n, A, generator=g), -9.0, 9.0)
    std = torch.exp(torch.clamp(torch.randn(n, A, generator=g), -5.0, 2.0))
    logits = 2.0 * torch.randn(n, 2, generator=g)
    mask = (torch.arange(n) % 3 != 1).int()
    env = torch.randint(0, 1 << 31, (n,), generator=g, dtype=torch.int64).to(torch.int32)
    t = torch.randint(0, 1 << 40, (n,), generator=g, dtype=torch.int64)
    return mean, std, logits, mask, env, t


def _run_sampler(seed, mean, std, logits, mask, env, t, advance_t=True, ldo=None):
    from tacorl_b200.rollout import policy_sample
    n, A = mean.shape
    out = torch.full((n, ldo or A + 1), SENTINEL, device=DEV)
    d = lambda x: None if x is None else x.to(DEV).contiguous()
    t_dev = d(t)
    policy_sample(d(mean), d(std), d(logits), d(mask), seed, d(env), t_dev, out, advance_t)
    torch.cuda.synchronize()
    return out.cpu(), t_dev.cpu()


def _check_sampler(seed, inputs, got, use_grip, use_mask, control=None):
    """Rows the mask writes against fp64 on the same uniforms, untouched rows, and t.  Returns (ok, worst)."""
    mean, std, logits, mask, env, t = inputs
    out, t_after = got
    n, A = mean.shape
    tt = t.numpy().astype(np.uint64) + (1 if control == "t_after_increment" else 0)
    ua, ub, ug = _uniforms(seed, tt, env.numpy().astype(np.uint64), A, use_grip,
                           draw0=0 if control == "draws_from_0" else RB.POLICY_DRAW0, swap=control == "ua_ub_swapped")
    written = (mask != 0) if (use_mask and control != "mask_ignored") else torch.ones(n, dtype=torch.bool)
    want = RB.tanh_normal_sample(mean, std, ua, ub)
    err = (out[:, :A].double() - want).abs()
    ok_cont = bool((err <= 1e-5 * (1.0 + want.abs()))[written].all())
    ok = ok_cont and bool((out[~written] == SENTINEL).all())
    if use_grip:
        sc = RB.gumbel_scores(logits, ug)
        near_tie = (sc[:, 1] - sc[:, 0]).abs() < 1e-5
        g_ok = (out[:, A].double() == RB.gripper_sample(logits, ug)) | near_tie
        ok = ok and bool(g_ok[written].all())
    else:
        ok = ok and bool((out[:, A] == SENTINEL).all())
    ok = ok and torch.equal(t_after, t + 1)
    return ok, float(err[written].max())


@pytest.mark.parametrize("use_grip", [True, False])
@pytest.mark.parametrize("use_mask", [True, False])
@pytest.mark.parametrize("n,A", [(1, 6), (5, 16), (64, 6), (64, 40)])
def test_sampler_against_fp64(n, A, use_mask, use_grip):
    seed = 0xC0FFEE12345
    inputs = _sampler_inputs(n, A, seed=n * 31 + A)
    mean, std, logits, mask, env, t = inputs
    got = _run_sampler(seed, mean, std, logits if use_grip else None, mask if use_mask else None, env, t)
    ok, worst = _check_sampler(seed, inputs, got, use_grip, use_mask)
    parity_report(f"rollout_sampler_n{n}_A{A}_mask{int(use_mask)}_grip{int(use_grip)}", {"ok": ok, "max_abs": worst})
    assert ok, worst
    for control in CONTROLS:
        if control == "mask_ignored" and not (use_mask and n > 1):
            continue
        assert not _check_sampler(seed, inputs, got, use_grip, use_mask, control)[0], control


def test_sampler_without_advance_and_with_a_row_stride():
    seed = 5
    mean, std, logits, mask, env, t = _sampler_inputs(8, 16, seed=2)
    out, t_after = _run_sampler(seed, mean, std, None, mask, env, t, advance_t=False, ldo=20)
    assert torch.equal(t_after, t)
    ref, _ = _run_sampler(seed, mean, std, None, mask, env, t)
    assert torch.equal(out[:, :16], ref[:, :16]) and bool((out[:, 16:] == SENTINEL).all())


def test_sampler_batch_invariance():
    """Every row of a 64-row call is bit-identical to the same row sampled alone."""
    seed = 77
    mean, std, logits, mask, env, t = _sampler_inputs(64, 16, seed=9)
    out, ta = _run_sampler(seed, mean, std, logits, mask, env, t)
    for r in range(64):
        one, t1 = _run_sampler(seed, mean[r:r + 1], std[r:r + 1], logits[r:r + 1], mask[r:r + 1], env[r:r + 1],
                               t[r:r + 1])
        assert torch.equal(one, out[r:r + 1]) and torch.equal(t1, ta[r:r + 1]), r


def test_sampler_distribution():
    """mean 0, std 1: atanh of 64 environments x 2000 steps is N(0, 1); gripper frequencies match softmax(logits)."""
    from scipy import stats
    from tacorl_b200.rollout import policy_sample
    n, A, steps = 64, 2, 2000
    mean, std = torch.zeros(n, A, device=DEV), torch.ones(n, A, device=DEV)
    logits = torch.tensor([0.4, -0.7], device=DEV).repeat(n, 1)
    env = torch.arange(n, device=DEV, dtype=torch.int32) * 7 + 3
    t = torch.zeros(n, device=DEV, dtype=torch.int64)
    out = torch.empty(steps, n, A + 1, device=DEV)
    for s in range(steps):
        policy_sample(mean, std, logits, None, 2024, env, t, out[s], advance_t=True)
    out = out.cpu().double()
    assert torch.equal(t.cpu(), torch.full((n,), steps, dtype=torch.int64))
    z = torch.atanh(out[..., :A]).reshape(-1).numpy()
    p = stats.kstest(z, "norm").pvalue
    p1 = float(torch.softmax(logits[0].cpu().double(), 0)[1])
    k = float((out[..., A] > 0).sum())
    N = steps * n
    sigma = (N * p1 * (1 - p1)) ** 0.5
    parity_report("rollout_sampler_distribution", {"ks_p": p, "grip_ones": k, "expected": N * p1, "sigma": sigma})
    assert p > 1e-3, p
    assert abs(k - N * p1) < 5 * sigma, (k, N * p1, sigma)
    assert set(out[..., A].unique().tolist()) == {-1.0, 1.0}


# ------------------------------------------------------------------------------------------------ whole policy
def _synth(module, seed):
    sd = S.synth_state_dict({k: list(v.shape) for k, v in module.state_dict().items()}, seed)
    module.load_state_dict(sd, strict=True)
    return module.to(DEV).eval(), sd


def _play_lmp(hidden, mods=("rgb_static",), latent=16, seed=22, precision="fp32"):
    from tacorl_b200 import ops
    ops.set_precision(precision)
    return _synth(build_play_lmp("tanh_net", mods, hidden, latent, 8, goal_modalities=mods), seed)


def _cql(seed=23, precision="fp32"):
    return _synth(build_cql_flat(precision), seed)


def _module(kind, hidden, mods, precision):
    latent = 32 if len(mods) > 1 else 16
    if kind == "play_lmp":
        return _play_lmp(hidden, mods, latent, precision=precision)
    if kind == "cql":
        return _cql(precision=precision)
    return _tacorl(hidden, mods, latent, precision=precision)


def _drive(policy, oracle, mods, n, steps, seed):
    """tests/test_gpu_rollout.py's _drive; flat CQL has no plan, so its replan events are skipped."""
    sz = _sizes(mods)
    got, want = [], []
    for s in range(steps):
        for kind, rows in _schedule(n, steps).get(s, []):
            if kind == "replan":
                if policy.kind != "cql":
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


CASES = [
    ("play_lmp", True, "fp32", ("rgb_static",)),
    ("play_lmp", True, "bf16", ("rgb_static",)),
    ("play_lmp", False, "fp32", ("rgb_static",)),
    ("play_lmp", False, "bf16", ("rgb_static",)),
    ("play_lmp", True, "fp32", ("rgb_static", "rgb_gripper")),
    ("play_lmp", False, "fp32", ("rgb_static", "rgb_gripper")),
    ("cql", True, "fp32", ("rgb_static",)),
    ("cql", True, "bf16", ("rgb_static",)),
    ("cql", False, "fp32", ("rgb_static",)),
    ("tacorl", False, "fp32", ("rgb_static",)),
    ("tacorl", False, "bf16", ("rgb_static",)),
]


@pytest.mark.parametrize("kind,deterministic,precision,mods", CASES)
def test_policy_matches_oracle(kind, deterministic, precision, mods):
    from tacorl_b200 import ops
    from tacorl_b200.rollout import RolloutPolicy
    hidden = 2048
    n, steps = (8, 24) if len(mods) == 1 else (4, 12)
    latent = 32 if len(mods) > 1 else 16
    m, sd = _module(kind, hidden, mods, precision)
    try:
        ops.set_precision(precision)
        ids = [100 + 3 * r for r in range(n)]
        policy = RolloutPolicy(m, n, seed=1234, env_ids=ids, deterministic=deterministic)
        oracle = RB.RolloutOracle(double_params(sd), n, hidden, latent, seed=1234, env_ids=ids, obs_mods=mods,
                                 goal_mods=mods, kind=kind, deterministic=deterministic)
        got, want = _drive(policy, oracle, mods, n, steps, seed=6)
        if precision == "fp32":
            assert_close(f"rollout actions {kind}", got, want, 1e-4, atol=1e-5)
        else:   # the criterion of tests/test_gpu_rollout.py: gripper exact, most dimensions close
            assert torch.equal(got[..., -1], want[..., -1])
            close = ((got[..., :6] - want[..., :6]).abs() < 5e-2).float().mean()
            assert close > 0.8, close
        parity_report(f"rollout_{kind}_{'det' if deterministic else 'sampled'}_{precision}_{len(mods)}view",
                      {"max_abs": float((got - want).abs().max()),
                       "launches": {str(k): v for k, v in policy.launches.items()}})
    finally:
        ops.set_precision("fp32")


@pytest.mark.parametrize("kind,deterministic", [("play_lmp", True), ("play_lmp", False), ("cql", True),
                                                ("cql", False), ("tacorl", False)])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_graph_replays_equal_eager_runs(kind, deterministic, precision):
    from tacorl_b200 import ops
    from tacorl_b200.rollout import RolloutPolicy
    mods = ("rgb_static",)
    m, _ = _module(kind, 2048, mods, precision)
    try:
        ops.set_precision(precision)
        a, _ = _drive(RolloutPolicy(m, 6, seed=9, deterministic=deterministic), None, mods, 6, 14, seed=2)
        b, _ = _drive(RolloutPolicy(m, 6, seed=9, deterministic=deterministic, use_graphs=False), None, mods, 6, 14,
                      seed=2)
        assert torch.equal(a, b)
    finally:
        ops.set_precision("fp32")


def test_sampled_and_deterministic_plans_differ_and_sampled_plans_follow_the_mask():
    """A sampled plan replaces only the flagged rows' plans, and differs from tanh(mean)."""
    from tacorl_b200 import ops
    from tacorl_b200.rollout import RolloutPolicy
    m, _ = _play_lmp(256)
    ops.set_precision("fp32")
    obs = {"rgb_static": S.synth_images((4, 3, 200, 200), 1, "o").to(DEV)}
    ps, pd = RolloutPolicy(m, 4, seed=3, deterministic=False), RolloutPolicy(m, 4, seed=3)
    for p in (ps, pd):
        p.reset(list(range(4)), obs)
        p.step(obs)
    assert not torch.allclose(ps.plan, pd.plan)
    before = ps.plan.clone()
    ps.replan([1])
    ps.step(obs)
    assert torch.equal(ps.plan[[0, 2, 3]], before[[0, 2, 3]]) and not torch.equal(ps.plan[1], before[1])


# library launches per replayed step and per replan step, as DESIGN.md section 16 states them
DESIGN_LAUNCHES = [
    ("play_lmp", True, "bf16", ("rgb_static",), 10, 12),
    ("play_lmp", False, "bf16", ("rgb_static",), 10, 13),
    ("play_lmp", True, "fp32", ("rgb_static",), 13, 15),
    ("play_lmp", False, "fp32", ("rgb_static",), 13, 16),
    ("play_lmp", True, "bf16", ("rgb_static", "rgb_gripper"), 17, 19),
    ("tacorl", False, "bf16", ("rgb_static",), 10, 20),
    ("tacorl", False, "fp32", ("rgb_static",), 13, 26),
    ("cql", True, "bf16", ("rgb_static",), 9, None),
    ("cql", False, "bf16", ("rgb_static",), 10, None),
    ("cql", True, "fp32", ("rgb_static",), 12, None),
    ("cql", False, "fp32", ("rgb_static",), 13, None),
]


@pytest.mark.parametrize("kind,deterministic,precision,mods,step,replan_step", DESIGN_LAUNCHES)
def test_launches_per_step_are_the_documented_ones(kind, deterministic, precision, mods, step, replan_step):
    from tacorl_b200 import ops
    from tacorl_b200.rollout import RolloutPolicy
    m, _ = _module(kind, 256, mods, precision)
    try:
        ops.set_precision(precision)
        p = RolloutPolicy(m, 4, seed=1, deterministic=deterministic)
        _drive(p, None, mods, 4, 3, seed=4)          # a replan step (not flat CQL), then plain steps
        parity_report(f"rollout_launches_{kind}_{'det' if deterministic else 'sampled'}_{precision}_{len(mods)}view",
                      {str(k): v for k, v in p.launches.items()})
        want = {(False, precision): step}
        if replan_step is not None:
            want[(True, precision)] = replan_step
        assert p.launches == want, p.launches
    finally:
        ops.set_precision("fp32")


@pytest.mark.parametrize("deterministic", [True, False])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_flat_cql_optimiser_built_after_capture_is_seen(precision, deterministic):
    """configure_optimizers after the capture moves the actor's parameters into a flat buffer: the policy recaptures,
    and a later torch edit reaches the replayed step exactly as it reaches an eager one."""
    from tacorl_b200 import ops
    from tacorl_b200.rollout import RolloutPolicy
    m, _ = _cql(precision=precision)
    try:
        ops.set_precision(precision)
        mods = ("rgb_static",)
        kw = dict(seed=8, deterministic=deterministic)
        pg, pe = RolloutPolicy(m, 3, **kw), RolloutPolicy(m, 3, use_graphs=False, **kw)
        a, b = _drive(pg, None, mods, 3, 4, seed=5)[0], _drive(pe, None, mods, 3, 4, seed=5)[0]
        assert torch.equal(a, b)
        captures = pg.captures
        w = m.actor.actor.policy.fc_mean.weight
        old_ptr = w.data_ptr()
        opts = m.configure_optimizers()
        assert w.data_ptr() != old_ptr
        obs = {"rgb_static": S.synth_images((3, 3, 200, 200), 5, "after").to(DEV)}
        g, e = pg.step(obs).cpu().clone(), pe.step(obs).cpu().clone()
        assert torch.equal(g, e) and pg.captures > captures
        saved = w.detach().clone()
        with torch.no_grad():
            w.mul_(3.0)
        g2, e2 = pg.step(obs).cpu().clone(), pe.step(obs).cpu().clone()
        assert torch.equal(g2, e2)
        # the edit is seen: with it undone, a replay at the t of the step before it gives that step's actions back
        assert len(opts) > 0
        with torch.no_grad():
            w.copy_(saved)
        pg.t.sub_(2)
        g3 = pg.step(obs).cpu().clone()
        assert torch.equal(g3, g) and not torch.equal(g2, g3)
    finally:
        ops.set_precision("fp32")


def test_flat_cql_rejects_replan():
    from tacorl_b200.rollout import RolloutPolicy
    m, _ = _cql()
    p = RolloutPolicy(m, 2)
    with pytest.raises(ValueError, match="flat CQL"):
        p.replan([0])
