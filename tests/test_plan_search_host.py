"""Host-side checks of the rollout policy's critic-guided plan search (DESIGN.md section 16.2): PlanSearch's and
RolloutPolicy's argument checks, the search's Philox mapping and its distance from the decoder's and the policy
sampler's draws, and the fp64 / fp32 oracle of tests/plan_search_oracle.py against hand-computed cases."""
import numpy as np
import pytest
import torch

from oracle import replay_oracle as RO
from tests import plan_search_oracle as PS
from tests.gpu_util import build_cql_flat, build_play_lmp, build_tacorl


def _u(w):
    return float(np.float32(int(w) >> 8) * np.float32(2.0 ** -24))


# ------------------------------------------------------------------------------------------------ arguments
def test_plan_search_settings_are_validated():
    from tacorl_b200.rollout import PlanSearch
    ok = PlanSearch(samples=128, elites=16, iterations=3, min_std=1e-3)
    assert (ok.samples, ok.elites, ok.iterations, ok.min_std) == (128, 16, 3, 1e-3)
    PlanSearch(samples=32, elites=32, iterations=1, min_std=1)
    PlanSearch(samples=np.int64(512), elites=1, iterations=8)
    bad = [dict(samples=0), dict(samples=16), dict(samples=48), dict(samples=544), dict(samples=128.0),
           dict(samples=True), dict(elites=0), dict(samples=64, elites=65), dict(elites=2.0), dict(elites=False),
           dict(iterations=0), dict(iterations=9), dict(iterations="3"), dict(iterations=True), dict(min_std=0.0),
           dict(min_std=-1e-3), dict(min_std=float("nan")), dict(min_std=float("inf")), dict(min_std=True),
           dict(min_std="0.1"), dict(min_std=1e-60)]
    for kw in bad:
        with pytest.raises(ValueError, match="PlanSearch"):
            PlanSearch(**kw)


def test_policy_refuses_plan_search_without_critics_or_plan():
    from tacorl_b200.rollout import PlanSearch, RolloutPolicy
    lmp = build_play_lmp("tanh_net", ("rgb_static",), 16, 8, 8, goal_modalities=("rgb_static",)).eval()
    with pytest.raises(ValueError, match="critic"):
        RolloutPolicy(lmp, 4, plan_search=PlanSearch())
    cql = build_cql_flat().eval()
    with pytest.raises(ValueError, match="no plan"):
        RolloutPolicy(cql, 4, plan_search=PlanSearch())
    t = build_tacorl(build_play_lmp("tanh_net", ("rgb_static",), 16, 8, 8, goal_modalities=("rgb_static",))).eval()
    with pytest.raises(ValueError, match="deterministic=False"):
        RolloutPolicy(t, 4, deterministic=False, plan_search=PlanSearch())
    with pytest.raises(ValueError, match="PlanSearch or None"):
        RolloutPolicy(t, 4, plan_search={"samples": 64})
    # accepted: what is left is the device (this module is on the CPU, and there is no CPU path)
    from tacorl_b200 import _lib
    with pytest.raises(_lib.TacorlLibraryError, match="CUDA"):
        RolloutPolicy(t, 4, plan_search=PlanSearch())


# ------------------------------------------------------------------------------------------------ noise
def test_search_uniforms_follow_the_stated_mapping():
    seed, t, env, K, P = 0x0123456789ABCDEF, (3 << 32) + 11, 42, 64, 16
    for k in (0, 2):
        ua, ub = PS.search_uniforms(seed, t, env, k, K, P)
        assert ua.shape == (K, P) and ua.dtype == np.float32
        for c, d in ((0, 0), (1, 5), (63, 15), (17, 3)):
            j = 256 + (k * K + c) * P + d
            w = RO.philox4x32_10(t & 0xFFFFFFFF, t >> 32, env, j, seed & 0xFFFFFFFF, seed >> 32)
            assert (float(ua[c, d]), float(ub[c, d])) == (_u(w[0]), _u(w[1])), (k, c, d)
    # rounds, environments and steps read different draws
    a = PS.search_uniforms(1, 0, 0, 0, 32, 8)[0]
    assert not np.array_equal(a, PS.search_uniforms(1, 0, 0, 1, 32, 8)[0])
    assert not np.array_equal(a, PS.search_uniforms(1, 0, 1, 0, 32, 8)[0])
    assert not np.array_equal(a, PS.search_uniforms(1, 1, 0, 0, 32, 8)[0])


def test_search_draws_stay_clear_of_the_decoder_and_the_policy_sampler():
    # the decoder reads draws 0..16, the policy sampler 32 + d for d <= A (A <= 64 continuous dimensions here)
    assert PS.SEARCH_DRAW0 > 32 + 64 + 1 > 16
    assert PS.SEARCH_DRAW0 + 8 * 512 * 64 < 2 ** 32


# ------------------------------------------------------------------------------------------------ the oracle
def test_candidates_and_score_by_hand():
    mu, sigma = torch.tensor([0.5, -0.25]), torch.tensor([2.0, 0.5])
    ua = np.array([[0.9, 0.9], [0.5, 0.0]], dtype=np.float32)
    ub = np.array([[0.3, 0.3], [0.25, 0.0]], dtype=np.float32)
    z0 = PS.candidates(mu, sigma, ua, ub, 0)
    assert z0[0].tolist() == [0.5, -0.25]               # round 0, candidate 0: the actor's plan itself
    e = np.sqrt(-2 * np.log(1 - np.float64(np.float32(0.5)))) * np.cos(2 * np.pi * 0.25)
    assert abs(float(z0[1, 0]) - (0.5 + 2.0 * e)) < 1e-15
    assert float(z0[1, 1]) == -0.25                     # u_a = 0: eps = 0
    z1 = PS.candidates(mu, sigma, ua, ub, 1)            # later rounds draw candidate 0 too
    e0 = np.sqrt(-2 * np.log(1 - np.float64(np.float32(0.9)))) * np.cos(2 * np.pi * np.float64(np.float32(0.3)))
    assert abs(float(z1[0, 0]) - (0.5 + 2.0 * e0)) < 1e-12
    # one-layer critics (the output layer only): Q = w . (e | tanh z) + b
    c1 = [(torch.tensor([[1.0, 2.0, 0.0]]), torch.tensor([0.5]))]
    c2 = [(torch.tensor([[0.0, 0.0, 1.0]]), torch.tensor([0.0]))]
    z = torch.tensor([[0.0, 0.0], [np.arctanh(0.5), np.arctanh(-0.5)]], dtype=torch.float64)
    s = PS.score([c1, c2], [torch.tensor([1.0]), torch.tensor([3.0])], z)
    # the inputs are (e | tanh z_0 | tanh z_1): Q1 = e + 2 tanh z_0 + 0.5, Q2 = tanh z_1
    q1 = torch.tensor([1.5, 1.5 + 1.0])
    q2 = torch.tensor([0.0, -0.5])
    assert torch.allclose(s, torch.minimum(q1, q2).double(), atol=1e-12)
    # a NaN critic output scores -inf
    cn = [(torch.tensor([[float("nan"), 0.0, 0.0]]), torch.tensor([0.0]))]
    assert PS.score([cn, c2], [torch.tensor([1.0]), torch.tensor([3.0])], z).tolist() == [-np.inf, -np.inf]
    # SiLU between layers
    two = [(torch.tensor([[1.0]]), torch.tensor([0.0])), (torch.tensor([[2.0]]), torch.tensor([1.0]))]
    x = torch.tensor([[0.7]], dtype=torch.float64)
    assert abs(float(PS.q_mlp(two, x)[0]) - (2 * 0.7 / (1 + np.exp(-0.7)) + 1)) < 1e-15


def test_elites_refit_and_best_by_hand():
    scores = np.array([1.0, 3.0, 3.0, -np.inf, 2.0, 3.0], dtype=np.float32)
    assert PS.elites(scores, 1) == [1]                  # ties -> the lower index
    assert PS.elites(scores, 3) == [1, 2, 5]
    assert PS.elites(scores, 4) == [1, 2, 4, 5]
    assert PS.elites(np.full(4, -np.inf), 2) == [0, 1]
    z = np.array([[0.0, 1.0], [1.0, 2.0], [3.0, 2.0], [9.0, 9.0], [5.0, 5.0], [2.0, -4.0]], dtype=np.float32)
    m, sd = PS.refit_f32(z, scores, 3, 1e-3)
    assert m.tolist() == [2.0, 0.0]
    assert np.allclose(sd, [np.sqrt(2.0 / 3.0), np.sqrt(24.0 / 3.0)], rtol=1e-7)
    m1, sd1 = PS.refit_f32(z, scores, 1, 0.125)         # one elite: std 0, floored
    assert m1.tolist() == [1.0, 2.0] and sd1.tolist() == [0.125, 0.125]
    # fp32 order: ((a + b) + c) / 3 with a rounding in between
    big = np.array([[1e8, 0], [1.0, 0], [1.0, 0]], dtype=np.float32)
    mb, _ = PS.refit_f32(big, np.array([3.0, 2.0, 1.0]), 3, 1e-3)
    assert mb[0] == np.float32((np.float32(np.float32(1e8) + np.float32(1.0)) + np.float32(1.0)) / np.float32(3))
    # best so far: strictly better replaces, ties keep the earlier round
    b = PS.best_update(None, 0, z, scores)
    assert b[1] == 3.0 and b[0].tolist() == [1.0, 2.0]
    b2 = PS.best_update(b, 1, z[::-1].copy(), scores[::-1].copy())
    assert b2[0].tolist() == [1.0, 2.0]
    b3 = PS.best_update(b, 2, z, scores + 1)
    assert b3[1] == 4.0


def test_whole_search_never_scores_below_the_actor_plan():
    g = torch.Generator().manual_seed(0)
    D, P, H = 6, 4, 16
    crit = [[(torch.randn(H, D + P, generator=g) * 0.5, torch.randn(H, generator=g) * 0.1),
             (torch.randn(H, H, generator=g) * 0.3, torch.randn(H, generator=g) * 0.1),
             (torch.randn(1, H, generator=g), torch.randn(1, generator=g))] for _ in range(2)]
    e = [torch.randn(D, generator=g), torch.randn(D, generator=g)]
    mu, sigma = torch.randn(P, generator=g), torch.rand(P, generator=g) + 0.1
    for K, E, I in ((32, 1, 1), (64, 8, 3), (32, 32, 2)):
        plan, value, trace = PS.search(crit, e, mu, sigma, K, E, I, 1e-3, seed=7, t=5, env_id=3)
        actor = float(PS.score(crit, e, mu[None].double())[0])
        assert abs(float(trace[0]["scores"][0]) - actor) < 1e-12     # candidate 0 of round 0 is the actor's plan
        assert value >= float(trace[0]["scores"][0])
        assert value == max(float(tr["scores"].max()) for tr in trace)
        assert len(trace) == I and plan.shape == (P,) and bool((plan.abs() < 1).all())
        if I > 1:         # later rounds start from the refit of the previous round's elites
            idx = PS.elites(trace[0]["scores"].numpy(), E)
            assert torch.allclose(trace[1]["mu"], trace[0]["z"][idx].mean(0))
