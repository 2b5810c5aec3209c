"""Host-side checks of the rollout policy's PlayLMP and flat-CQL support and its sampler: the policy uniforms follow the
stated Philox mapping and stay clear of the decoder's draws, the oracle's PlayLMP and flat-CQL rollouts stepped frame by
frame with restarts equal whole segments, and RolloutPolicy's argument checks for the new module kinds."""
import numpy as np
import pytest
import torch

from oracle import ref_loader_cfg as RC
from oracle import replay_oracle as RO
from oracle import rollout_oracle as R
from oracle import synth as S
from tests import rollout_baselines_oracle as RB
from oracle import tacorl_oracle as O
from tests.gpu_util import build_cql_flat, build_play_lmp, double_params

KAT = [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]     # Random123: counter (0, 0, 0, 0), key (0, 0)


def _u(w):
    return float(np.float32(int(w) >> 8) * np.float32(2.0 ** -24))


def test_policy_uniforms_follow_the_stated_mapping():
    seed, t, env, A = 0x0123456789ABCDEF, (5 << 32) + 17, 9, 6
    ua, ub, ug = RB.policy_uniforms(seed, t, env, A, True)
    assert ua.shape == (A,) and ub.shape == (A,) and ug.shape == (2,) and ua.dtype == torch.float32
    for d in range(A + 1):
        w = RO.philox4x32_10(t & 0xFFFFFFFF, t >> 32, env, 32 + d, seed & 0xFFFFFFFF, seed >> 32)
        got = (float(ua[d]), float(ub[d])) if d < A else (float(ug[0]), float(ug[1]))
        assert got == (_u(w[0]), _u(w[1])), d
    # no gripper: the same continuous draws
    ua2, ub2, none = RB.policy_uniforms(seed, t, env, A, False)
    assert none is None and torch.equal(ua2, ua) and torch.equal(ub2, ub)
    # broadcast over steps and environments
    a, b, g = RB.policy_uniforms(3, np.arange(4)[:, None], np.array([0, 1, 2])[None, :], 16, True)
    assert a.shape == (4, 3, 16) and g.shape == (4, 3, 2)
    assert torch.equal(a[2, 1], RB.policy_uniforms(3, 2, 1, 16, True)[0])
    assert not torch.equal(a[0, 0], a[0, 1]) and not torch.equal(a[0, 0], a[1, 0])


def test_policy_uniforms_rest_on_the_pinned_philox_known_answers():
    assert [int(w) for w in RO.philox4x32_10(0, 0, 0, 0, 0, 0)] == KAT
    # draw 32 + d is the generator's block at counter word 3 = 32 + d: the known answer's words at draw 0, shifted
    ua, ub, _ = RB.policy_uniforms(0, 0, 0, 1, False)
    w = RO.philox4x32_10(0, 0, 0, 32, 0, 0)
    assert (float(ua[0]), float(ub[0])) == (_u(w[0]), _u(w[1]))
    assert float(ua[0]) != _u(KAT[0])


def test_policy_draws_never_meet_the_decoders():
    decoder = set(range((R.N_UNIFORMS + 3) // 4))          # draws 0..16
    assert max(decoder) == 16
    for A in (1, 6, 16, 256, 1024):
        assert not decoder & set(range(RB.POLICY_DRAW0, RB.POLICY_DRAW0 + A + 1))
    # so a sampled plan and the decoder step of the same t read different words
    u1, u2 = R.uniforms(7, 3, 4)
    ua, ub, _ = RB.policy_uniforms(7, 3, 4, 16, False)
    dec = set(torch.cat([u1.reshape(-1), u2]).tolist())
    assert not dec & set(torch.cat([ua, ub]).tolist())


def test_sampling_formulas():
    mean, std = torch.tensor([0.3, -1.0], dtype=torch.float64), torch.tensor([0.5, 2.0], dtype=torch.float64)
    ua, ub = torch.tensor([0.25, 0.0]), torch.tensor([0.125, 0.5])
    z = np.sqrt(-2 * np.log(1 - np.array([0.25, 0.0]))) * np.cos(2 * np.pi * np.array([0.125, 0.5]))
    want = np.tanh(np.array([0.3, -1.0]) + np.array([0.5, 2.0]) * z)
    assert np.allclose(RB.tanh_normal_sample(mean, std, ua, ub).numpy(), want, rtol=0, atol=1e-15)
    logits = torch.tensor([[0.0, 0.0], [0.0, 0.0], [1.0, -1.0]])
    u = torch.tensor([[0.5, 0.5], [0.0, 0.5], [0.5, 0.0]])
    # tie -> class 0; u = 0 scores -inf
    assert RB.gripper_sample(logits, u).tolist() == [-1.0, 1.0, -1.0]


# ------------------------------------------------------------------------------------------------ oracle rollouts
IMG = 48


def _play_lmp_params(hidden=16, latent=8, seed=3):
    lmp = build_play_lmp("tanh_net", ("rgb_static",), hidden, latent, 8, goal_modalities=("rgb_static",))
    sd = S.synth_state_dict({k: list(v.shape) for k, v in lmp.state_dict().items()}, seed)
    return double_params(sd)


def _cql_params(seed=4):
    m = build_cql_flat()
    sd = S.synth_state_dict({k: list(v.shape) for k, v in m.state_dict().items()}, seed)
    return double_params(sd)


def _img(tag, n=1):
    return S.synth_images((n, 3, IMG, IMG), 5, tag).double()


@pytest.mark.parametrize("deterministic", [True, False])
def test_play_lmp_oracle_stepping_with_restarts_equals_whole_segments(deterministic):
    """Frame by frame with a replan at step 4 == the plan proposal at each segment's first frame, then
    action_decoder_forward over the segment from h = 0, with the same uniforms."""
    P = _play_lmp_params()
    T, segs, env, seed = 7, [(0, 4), (4, 7)], 3, 11
    frames = [_img(f"f{s}") for s in range(T)]
    goal = _img("goal")
    orc = RB.RolloutOracle(P, 1, 16, 8, seed=seed, env_ids=[env], kind="play_lmp", deterministic=deterministic)
    orc.reset([0], {"rgb_static": goal})
    stepped = []
    for s in range(T):
        if s == 4:
            orc.replan([0])
        stepped.append(orc.step({"rgb_static": frames[s]})[0][0])
    stepped = torch.stack(stepped)
    enc = lambda x: O.lmp_encoder(P, "perceptual_encoder.networks.rgb_static.", x)
    g = O.goal_encoder(P, "goal_encoder.", enc(goal))
    u1, u2 = R.uniforms(seed, np.arange(T), env)
    whole = []
    for a, b in segs:
        mu, std = O.mlp_policy(P, "plan_proposal.policy.", torch.cat([enc(frames[a]), g], -1))
        if deterministic:
            plan = torch.tanh(mu)
        else:
            ua, ub, _ = RB.policy_uniforms(seed, a, env, 8, False)
            plan = RB.tanh_normal_sample(mu, std, ua, ub)
        emb = torch.cat([enc(frames[s]) for s in range(a, b)], 0)[None]
        lp, ls, mm, grip, _ = O.action_decoder_forward(P, "action_decoder.", plan, emb)
        whole.append(O.dlm_sample(lp, ls, mm, grip, u1[a:b][None].double(), u2[a:b][None].double())[0])
    whole = torch.cat(whole)
    assert torch.allclose(stepped, whole, rtol=1e-12, atol=1e-12)
    # the sampled plan is not tanh(mean)
    if not deterministic:
        det = RB.RolloutOracle(P, 1, 16, 8, seed=seed, env_ids=[env], kind="play_lmp")
        det.reset([0], {"rgb_static": goal})
        assert not torch.allclose(det.step({"rgb_static": frames[0]})[0][0], stepped[0])


@pytest.mark.parametrize("deterministic", [True, False])
def test_cql_oracle_stepping_with_restarts_equals_whole_segments(deterministic):
    """Frame by frame, with a reset (t back to 0, new goal) at step 4 == the actor over each segment's frames at once,
    with the uniforms of steps 0.. of each segment."""
    P = _cql_params()
    T, segs, env, seed = 7, [(0, 4), (4, 7)], 5, 12
    frames = [_img(f"c{s}") for s in range(T)]
    goals = [_img("g0"), _img("g1")]
    orc = RB.RolloutOracle(P, 1, 16, 8, seed=seed, env_ids=[env], kind="cql", deterministic=deterministic)
    stepped = []
    for s in range(T):
        if s in (0, 4):
            orc.reset([0], {"rgb_static": goals[s // 4]})
        stepped.append(orc.step({"rgb_static": frames[s]})[0][0])
    stepped = torch.stack(stepped)
    whole = []
    for k, (a, b) in enumerate(segs):
        obs = torch.cat(frames[a:b], 0)
        x = O.visual_emb(P, "actor.", {"rgb_static": obs}, {"rgb_static": goals[k].expand(b - a, -1, -1, -1)})
        mu, std, lg = O.mlp_policy_gripper(P, "actor.actor.policy.", x)
        if deterministic:
            whole.append(torch.cat([torch.tanh(mu), O.gumbel_argmax(lg, torch.full_like(lg, 0.5), False)
                                    .double()[:, None] * 2 - 1], -1))
        else:
            ua, ub, ug = RB.policy_uniforms(seed, np.arange(b - a), env, 6, True)
            whole.append(torch.cat([RB.tanh_normal_sample(mu, std, ua, ub), RB.gripper_sample(lg, ug)[:, None]], -1))
    whole = torch.cat(whole)
    assert stepped.shape == (T, 7)
    assert torch.allclose(stepped, whole, rtol=1e-12, atol=1e-12)
    if not deterministic:       # after the reset the noise repeats: t restarted at 0
        ua0 = RB.policy_uniforms(seed, 0, env, 6, True)
        assert torch.equal(ua0[0], RB.policy_uniforms(seed, np.arange(3), env, 6, True)[0][0])


# ------------------------------------------------------------------------------------------------ argument checks
def _modules():
    lmp = build_play_lmp("tanh_net", ("rgb_static",), 64, 16, 8, goal_modalities=("rgb_static",))
    return {"play_lmp": lmp, "cql": build_cql_flat()}


def test_play_lmp_and_flat_cql_are_accepted_in_eval_mode_and_refused_in_train_mode():
    from tacorl_b200 import _lib
    from tacorl_b200.rollout import RolloutPolicy, _module_kind
    for kind, m in _modules().items():
        assert _module_kind(m) == kind
        with pytest.raises(ValueError, match="eval"):
            RolloutPolicy(m.train(), 4)
        # accepted: what is left is the device (this module is on the CPU, and there is no CPU path)
        for det in (True, False):
            with pytest.raises(_lib.TacorlLibraryError, match="CUDA"):
                RolloutPolicy(m.eval(), 4, deterministic=det)


def test_continuous_gripper_flat_cql_is_refused():
    from tacorl_b200.rollout import RolloutPolicy
    m = build_cql_flat(actor=RC.actor_cfg()).eval()
    assert not m.actor.discrete_gripper
    with pytest.raises(ValueError, match="discrete"):
        RolloutPolicy(m, 4)


def test_replan_on_flat_cql_raises():
    from tacorl_b200.rollout import RolloutPolicy
    p = object.__new__(RolloutPolicy)
    p._dec, p.n = None, 4
    with pytest.raises(ValueError, match="flat CQL"):
        p.replan([0])


@pytest.mark.parametrize("bad", [1, 0, None, "yes", np.bool_(True)])
def test_non_bool_deterministic_is_refused(bad):
    from tacorl_b200.rollout import RolloutPolicy
    for m in _modules().values():
        with pytest.raises(ValueError, match="deterministic"):
            RolloutPolicy(m.eval(), 4, deterministic=bad)


def test_unsupported_modules_still_name_taco_rl():
    from tacorl_b200.rollout import RolloutPolicy
    with pytest.raises(ValueError, match="TACO-RL"):
        RolloutPolicy(torch.nn.Linear(2, 2).eval(), 4)
