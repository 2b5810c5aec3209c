"""GPU tests of the rollout policy's critic-guided plan search (tacorl_b200/rollout.py PlanSearch / plan_search,
csrc/plan_search.cu, DESIGN.md section 16.2): the Philox draws bit for bit, selection / refit / best plan recomputed
from the device's own candidates and scores, the scores against fp64, batch invariance, the search never scoring
below the actor's plan, graph replays against eager steps, and the library launches of a search replan step."""
import numpy as np
import pytest
import torch

from oracle import synth as S
from tests import plan_search_oracle as PS
from tests.gpu_util import DEV, build_play_lmp, build_tacorl, parity_report

pytestmark = pytest.mark.gpu

P_DIM, DO, DG, HID = 16, 32, 32, 256


def _critics(D, P, H, layers=3, seed=0):
    from tacorl_b200.networks.actor_critic.critic import MLPQNetwork
    torch.manual_seed(seed)
    qs = [MLPQNetwork(D + P, H, layers) for _ in range(2)]
    with torch.no_grad():          # an output layer at a scale where the candidates' scores spread
        for j, q in enumerate(qs):
            q.out.weight.normal_(0.0, 0.3)
            q.out.bias.fill_(0.1 * j)
    return [q.to(DEV).eval() for q in qs]


def _inputs(n, seed, P=P_DIM, Do=DO, Dg=DG):
    g = torch.Generator().manual_seed(seed)
    eo = [torch.randn(n, Do, generator=g) for _ in range(2)]
    eg = [torch.randn(n, Dg, generator=g) for _ in range(2)]
    mean = torch.randn(n, P, generator=g) * 0.5
    std = torch.rand(n, P, generator=g) * 0.5 + 0.05
    env = torch.randint(0, 1 << 20, (n,), generator=g, dtype=torch.int32)
    t = torch.randint(0, 1 << 40, (n,), generator=g, dtype=torch.int64)
    restart = (torch.arange(n) % 4 != 3).int()
    return dict(eo=eo, eg=eg, mean=mean, std=std, env=env, t=t, restart=restart)


def _run(qs, x, ps, seed, trace=True, uniforms=False):
    from tacorl_b200.rollout import SearchBuffers, plan_search
    n, P = x["mean"].shape
    H = qs[0].fc_layers[0].weight.shape[0]
    d = {k: ([v.to(DEV) for v in x[k]] if isinstance(x[k], list) else x[k].to(DEV).contiguous()) for k in x}
    bufs = SearchBuffers(n, ps.samples, P, H, DEV)
    plan = torch.full((n, P), 7.0, device=DEV)
    value = torch.full((n,), 7.0, device=DEV)
    tr, us = ([] if trace else None), ([] if uniforms else None)
    plan_search(qs, d["eo"], d["eg"], d["mean"], d["std"], ps, seed, d["env"], d["t"], d["restart"], plan, value, bufs,
                trace=tr, uniforms=us)
    torch.cuda.synchronize()
    cpu = lambda v: [{k: a.cpu() for k, a in r.items()} for r in v] if v is not None else None
    return plan.cpu(), value.cpu(), cpu(tr), ([u.cpu() for u in us] if us is not None else None), bufs


def _layers64(q):
    return [(fc.weight.detach().double().cpu(), fc.bias.detach().double().cpu()) for fc in q.fc_layers] + \
           [(q.out.weight.detach().double().cpu(), q.out.bias.detach().double().cpu())]


def _e(x, i):
    return [torch.cat([x["eo"][j][i], x["eg"][j][i]]).double() for j in range(2)]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_philox_draws_and_candidates(precision):
    from tacorl_b200 import ops
    from tacorl_b200.rollout import PlanSearch
    ops.set_precision(precision)
    try:
        qs = _critics(DO + DG, P_DIM, HID)
        x = _inputs(3, seed=1)
        ps = PlanSearch(samples=64, elites=8, iterations=2)
        seed = 0xFEEDFACE12345678
        _, _, tr, us, _ = _run(qs, x, ps, seed, uniforms=True)
        for k in range(ps.iterations):
            u = us[k].view(3, 64, P_DIM, 2)
            z = tr[k]["z"].view(3, 64, P_DIM)
            for i in range(3):
                ua, ub = PS.search_uniforms(seed, int(x["t"][i]), int(x["env"][i]), k, 64, P_DIM)
                assert np.array_equal(u[i, ..., 0].numpy(), ua) and np.array_equal(u[i, ..., 1].numpy(), ub), (k, i)
                mu, sg = (x["mean"][i], x["std"][i]) if k == 0 else (tr[k - 1]["mu"][i], tr[k - 1]["sigma"][i])
                want = PS.candidates(mu, sg, ua, ub, k)
                assert torch.allclose(z[i].double(), want, rtol=1e-5, atol=1e-5), (k, i)
                if k == 0:
                    assert torch.equal(z[i, 0], x["mean"][i])          # the actor's deterministic plan, exactly
    finally:
        ops.set_precision("fp32")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("K,E,I", [(64, 8, 3), (32, 1, 2), (128, 128, 1)])
def test_selection_refit_and_best_from_device_scores(precision, K, E, I):
    from tacorl_b200 import ops
    from tacorl_b200.rollout import PlanSearch
    ops.set_precision(precision)
    try:
        qs = _critics(DO + DG, P_DIM, HID, seed=2)
        n = 5
        x = _inputs(n, seed=K + E)
        ps = PlanSearch(samples=K, elites=E, iterations=I, min_std=1e-2)
        plan, value, tr, _, bufs = _run(qs, x, ps, 99)
        for i in range(n):
            best = None
            for k in range(I):
                z = tr[k]["z"].view(n, K, P_DIM)[i].numpy()
                s = tr[k]["scores"][i].numpy()
                m, sd = PS.refit_f32(z, s, E, ps.min_std)
                assert np.array_equal(tr[k]["mu"][i].numpy(), m), (i, k)
                assert np.array_equal(tr[k]["sigma"][i].numpy(), sd), (i, k)
                best = PS.best_update(best, k, z, s)
                assert np.array_equal(tr[k]["best_z"][i].numpy(), best[0]) and float(tr[k]["best_s"][i]) == best[1]
            if int(x["restart"][i]):
                assert float(value[i]) == best[1]
                assert torch.allclose(plan[i], torch.tanh(bufs.best_z[i]).cpu(), rtol=0, atol=1e-6)
            else:                      # a row not flagged keeps its plan and value
                assert bool((plan[i] == 7.0).all()) and float(value[i]) == 7.0
    finally:
        ops.set_precision("fp32")


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_scores_against_fp64(precision, tol):
    from tacorl_b200 import ops
    from tacorl_b200.rollout import PlanSearch
    ops.set_precision(precision)
    try:
        qs = _critics(DO + DG, P_DIM, HID, seed=3)
        n = 4
        x = _inputs(n, seed=5)
        ps = PlanSearch(samples=64, elites=8, iterations=2)
        _, _, tr, _, _ = _run(qs, x, ps, 3)
        crit = [_layers64(q) for q in qs]
        worst = 0.0
        for k in range(ps.iterations):
            for i in range(n):
                z = tr[k]["z"].view(n, 64, P_DIM)[i].double()
                want = PS.score(crit, _e(x, i), z)
                got = tr[k]["scores"][i].double()
                err = float((got - want).abs().max() / max(1.0, float(want.abs().max())))
                worst = max(worst, err)
        parity_report(f"plan_search_scores_{precision}", {"worst_rel": worst, "tol": tol})
        assert worst <= tol, worst
    finally:
        ops.set_precision("fp32")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_batch_invariance(precision):
    """A row searched alone and the same row among 64, at several positions: bit-identical plans, values, and the
    actions of the decoder step that follows."""
    from tacorl_b200 import ops
    from tacorl_b200.networks.action_decoders.action_decoder_logistic import ActionDecoderLogistic
    from tacorl_b200.rollout import PlanSearch, decoder_step
    ops.set_precision(precision)
    try:
        qs = _critics(DO + DG, P_DIM, HID, seed=4)
        torch.manual_seed(4)
        dec = ActionDecoderLogistic(state_dim=32, latent_plan_dim=P_DIM, hidden_size=256).to(DEV).eval()
        ps = PlanSearch(samples=64, elites=8, iterations=3)
        one = _inputs(1, seed=11)
        one["restart"][:] = 1

        def act(plan, n):
            emb = torch.ones(n, 32, device=DEV) * 0.1
            hidden = torch.zeros(2, n, 256, device=DEV)
            acts = torch.empty(n, 7, device=DEV)
            env = torch.full((n,), 5, dtype=torch.int32, device=DEV)
            decoder_step(dec, plan.to(DEV), emb, hidden, torch.ones(n, dtype=torch.int32, device=DEV), 3, env,
                         torch.zeros(n, dtype=torch.int64, device=DEV), acts)
            return acts.cpu()

        p1, v1, _, _, _ = _run(qs, one, ps, 21, trace=False)
        a1 = act(p1, 1)
        for pos in (0, 17, 63):
            many = _inputs(64, seed=12 + pos)
            many["restart"][:] = 1
            for k in many:
                if isinstance(many[k], list):
                    for j in range(2):
                        many[k][j][pos] = one[k][j][0]
                else:
                    many[k][pos] = one[k][0]
            pm, vm, _, _, _ = _run(qs, many, ps, 21, trace=False)
            assert torch.equal(pm[pos], p1[0]) and torch.equal(vm[pos], v1[0]), pos
            assert torch.equal(act(pm, 64)[pos], a1[0]), pos
    finally:
        ops.set_precision("fp32")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_value_never_below_the_actor_plan(precision):
    from tacorl_b200 import ops
    from tacorl_b200.rollout import PlanSearch
    ops.set_precision(precision)
    try:
        qs = _critics(DO + DG, P_DIM, HID, seed=6)
        n = 16
        x = _inputs(n, seed=8)
        x["restart"][:] = 1
        for ps in (PlanSearch(samples=32, elites=4, iterations=1), PlanSearch(samples=128, elites=16, iterations=3)):
            _, value, tr, _, _ = _run(qs, x, ps, 8)
            actor = tr[0]["scores"][:, 0]          # candidate (0, 0): the actor's tanh(mean), scored by both kernels
            assert bool((value >= actor).all())
            assert float((value - actor).max()) > 0          # and the search finds better plans somewhere
    finally:
        ops.set_precision("fp32")


# ------------------------------------------------------------------------------------------------ the policy
def _tacorl(precision, seed=21):
    lmp = build_play_lmp("tanh_net", ("rgb_static",), 256, P_DIM, 8, goal_modalities=("rgb_static",))
    t = build_tacorl(lmp, precision)
    sd = S.synth_state_dict({k: list(v.shape) for k, v in t.state_dict().items()}, seed)
    t.load_state_dict(sd, strict=True)
    with torch.no_grad():
        for q in (t.q1, t.q2):
            q.critic.Q.out.weight.normal_(0.0, 0.3)
    return t.to(DEV).eval()


def _drive(policy, n, steps, seed):
    got, values = [], []
    for s in range(steps):
        if s == 0:
            policy.reset(list(range(n)), {"rgb_static": S.synth_images((n, 3, 200, 200), seed, "goal").to(DEV)})
        elif s % 4 == 0:
            policy.replan([r for r in range(n) if (r + s) % 2 == 0])
        obs = {"rgb_static": S.synth_images((n, 3, 200, 200), seed, f"obs{s}").to(DEV)}
        got.append(policy.step(obs).cpu().clone())
        values.append(policy.plan_value.cpu().clone() if policy.plan_value is not None else None)
    return torch.stack(got), values


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_graph_replay_equals_eager_step(precision):
    from tacorl_b200 import ops
    from tacorl_b200.rollout import PlanSearch, RolloutPolicy
    t = _tacorl(precision)
    try:
        ops.set_precision(precision)
        ps = PlanSearch(samples=64, elites=8, iterations=2)
        a, va = _drive(RolloutPolicy(t, 6, seed=9, plan_search=ps), 6, 10, seed=2)
        b, vb = _drive(RolloutPolicy(t, 6, seed=9, plan_search=ps, use_graphs=False), 6, 10, seed=2)
        assert torch.equal(a, b)
        assert all(torch.equal(x, y) for x, y in zip(va, vb))
        assert not bool(torch.isnan(va[-1]).any())
        # the search changes the plans: the actions differ from the actor's plan
        c, _ = _drive(RolloutPolicy(t, 6, seed=9), 6, 10, seed=2)
        assert not torch.equal(a, c)
    finally:
        ops.set_precision("fp32")


def test_policy_value_is_the_critics_min_of_its_plan():
    """fp32: plan_value equals min(Q1, Q2) of the chosen plan as the module's own critic forward computes it on
    cat(encoder_qj(obs), goal_encoder_qj(encoder_qj(goal))), and is never below the actor's plan's score."""
    from tacorl_b200.rollout import PlanSearch, RolloutPolicy
    t = _tacorl("fp32", seed=5)
    n = 4
    p = RolloutPolicy(t, n, seed=3, plan_search=PlanSearch(samples=128, elites=16, iterations=1))
    goal = {"rgb_static": S.synth_images((n, 3, 200, 200), 1, "g").to(DEV)}
    obs = {"rgb_static": S.synth_images((n, 3, 200, 200), 1, "o").to(DEV)}
    p.reset(list(range(n)), goal)
    p.step(obs)
    with torch.no_grad():
        q = []
        for c in (t.q1, t.q2):
            e = c.encoder.get_state_from_observation(observation=obs, modalities=c.env_modalities)
            g = c.goal_encoder(c.encoder.get_state_from_observation(observation=goal, modalities=c.goal_modalities))
            q.append(t._q_mlp(c.critic.Q, torch.cat([e, g], -1), p.plan).reshape(-1))
        want = torch.minimum(q[0], q[1])
    assert torch.allclose(p.plan_value, want, rtol=1e-4, atol=1e-4), (p.plan_value, want)
    actor = p._search_bufs.scores[:, 0]             # one round: candidate 0 is the actor's plan
    assert bool((p.plan_value >= actor).all())


@pytest.mark.parametrize("precision,optimiser", [("fp32", False), ("bf16", False), ("bf16", True)])
def test_launches_of_a_search_replan_step(precision, optimiser):
    """The replan graph adds one encoder pass per critic and, per round, sample_l0 + (L - 1) hidden layers of both
    critics (+ a bf16 cast of each weight without a bf16 copy) + select; the plain step's graph is unchanged."""
    from tacorl_b200 import _lib, ops
    from tacorl_b200.rollout import PlanSearch, RolloutPolicy
    t = _tacorl(precision)
    try:
        ops.set_precision(precision)
        opts = t.configure_optimizers() if optimiser else None
        ps = PlanSearch(samples=64, elites=8, iterations=3)
        base = RolloutPolicy(t, 4, seed=1)
        srch = RolloutPolicy(t, 4, seed=1, plan_search=ps)
        _drive(base, 4, 3, seed=4)
        _drive(srch, 4, 3, seed=4)
        obs = {"rgb_static": S.synth_images((4, 3, 200, 200), 4, "obs0").to(DEV)}
        with torch.no_grad():
            t.q1.encoder.get_state_from_observation(observation=obs, modalities=t.q1.env_modalities)
            n0 = _lib.launch_count()
            t.q1.encoder.get_state_from_observation(observation=obs, modalities=t.q1.env_modalities)
            enc = _lib.launch_count() - n0
        nl = len(t.q1.critic.Q.fc_layers)
        # bf16: a hidden weight without a 16-byte aligned bf16 copy is cast first
        staged = lambda w: precision == "bf16" and (ops.shadow_of(w) is None or ops.shadow_of(w).data_ptr() % 16 != 0)
        per_round = 2 + sum(1 + int(staged(q.critic.Q.fc_layers[l].weight)) for q in (t.q1, t.q2) for l in range(1, nl))
        if not optimiser:
            assert per_round == 2 + 2 * (nl - 1) * (2 if precision == "bf16" else 1)
        assert srch.launches[(False, precision)] == base.launches[(False, precision)]
        assert srch.launches[(True, precision)] == base.launches[(True, precision)] + 2 * enc + ps.iterations * per_round
        parity_report(f"plan_search_launches_{precision}_{'opt' if optimiser else 'noopt'}",
                      {"replan_step": srch.launches[(True, precision)], "step": srch.launches[(False, precision)],
                       "base_replan_step": base.launches[(True, precision)], "encoder_pass": enc,
                       "per_round": per_round})
        assert opts is None or len(opts) > 0
    finally:
        ops.set_precision("fp32")
