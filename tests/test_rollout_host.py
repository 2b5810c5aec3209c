"""Host-side checks of the batched rollout policy: the oracle's counter-based uniforms follow the stated mapping, the
oracle's per-frame stepping with restarts equals the decoder run over whole segments, and RolloutPolicy rejects
malformed arguments before touching a device."""
import numpy as np
import pytest
import torch

from oracle import replay_oracle as RO
from oracle import rollout_oracle as R
from oracle import synth as S
from oracle import tacorl_oracle as O


def test_uniforms_follow_the_stated_philox_mapping():
    seed, t, env = 0x0123456789ABCDEF, (5 << 32) + 17, 9
    u1, u2 = R.uniforms(seed, t, env)
    assert u1.shape == (6, 10) and u2.shape == (6,) and u1.dtype == torch.float32
    flat = torch.cat([u1.reshape(-1), u2])
    for i in range(66):
        w = RO.philox4x32_10(t & 0xFFFFFFFF, t >> 32, env, i // 4, seed & 0xFFFFFFFF, seed >> 32)[i % 4]
        assert float(flat[i]) == float(np.float32(int(w) >> 8) * np.float32(2.0 ** -24)), i
    assert 0.0 <= float(flat.min()) and float(flat.max()) < 1.0


def test_uniforms_rest_on_the_pinned_philox_known_answers():
    # counter (0, 0, 0, 0), key (0, 0): the Random123 known answer test_replay_host.py pins
    kat = [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    u1, _ = R.uniforms(0, 0, 0)
    assert [float(v) for v in u1[0, :4]] == [(w >> 8) * 2.0 ** -24 for w in kat]


def test_uniforms_are_per_environment_and_per_step():
    u_a, _ = R.uniforms(3, np.arange(4)[:, None], np.array([0, 1, 2])[None, :])
    assert u_a.shape == (4, 3, 6, 10)
    for s in range(4):
        for e in range(3):
            assert torch.equal(u_a[s, e], R.uniforms(3, s, e)[0])
    assert not torch.equal(u_a[0, 0], u_a[0, 1]) and not torch.equal(u_a[0, 0], u_a[1, 0])
    assert not torch.equal(R.uniforms(3, 0, 0)[0], R.uniforms(4, 0, 0)[0])


def _decoder_params(hidden=16, latent=8, state=12, seed=3):
    shapes = {}
    I = latent + state
    for l in range(2):
        shapes[f"action_decoder.rnn.weight_ih_l{l}"] = [hidden, I if l == 0 else hidden]
        shapes[f"action_decoder.rnn.weight_hh_l{l}"] = [hidden, hidden]
        shapes[f"action_decoder.rnn.bias_ih_l{l}"] = [hidden]
        shapes[f"action_decoder.rnn.bias_hh_l{l}"] = [hidden]
    for k in ("prob_fc", "mean_fc", "log_scale_fc"):
        shapes[f"action_decoder.{k}.weight"], shapes[f"action_decoder.{k}.bias"] = [60, hidden], [60]
    shapes["action_decoder.gripper_fc.weight"], shapes["action_decoder.gripper_fc.bias"] = [2, hidden], [2]
    sd = S.synth_state_dict(shapes, seed)
    return {k: v.double() for k, v in sd.items()}


def test_stepping_with_restarts_equals_whole_segments():
    """One frame at a time, a restart zeroing the hidden state, == action_decoder_forward over each segment from h = 0,
    with the same uniforms."""
    P = _decoder_params()
    g = torch.Generator().manual_seed(0)
    T, segs = 9, [(0, 4), (4, 9)]          # a restart (replan) at step 4
    emb = torch.randn(1, T, 12, generator=g, dtype=torch.float64)
    plans = [torch.randn(1, 8, generator=g, dtype=torch.float64) for _ in segs]
    u1, u2 = R.uniforms(11, np.arange(T), 2)
    u1, u2 = u1.double(), u2.double()
    h = torch.zeros(2, 1, 16, dtype=torch.float64)
    stepped = []
    for s in range(T):
        k = 0 if s < 4 else 1
        if s == 4:
            h = torch.zeros_like(h)
        heads, h = R.decoder_step(P, plans[k], emb[:, s], h)
        stepped.append(R.sample(heads, u1[s][None], u2[s][None])[0])
    stepped = torch.stack(stepped)
    whole = []
    for k, (a, b) in enumerate(segs):
        lp, ls, mm, grip, _ = O.action_decoder_forward(P, "action_decoder.", plans[k], emb[:, a:b])
        whole.append(O.dlm_sample(lp, ls, mm, grip, u1[a:b][None], u2[a:b][None])[0])
    whole = torch.cat(whole)
    assert torch.allclose(stepped, whole, rtol=1e-12, atol=1e-12)
    # without the restart the second segment differs (the recurrence carries over)
    heads, _ = R.decoder_step(P, plans[1], emb[:, 4], h)
    assert not torch.allclose(R.sample(heads, u1[4][None], u2[4][None])[0], whole[4])


class _Fake(torch.nn.Module):
    """Just enough of a TACO-RL module for the argument checks that run before any device work."""

    def __init__(self):
        super().__init__()
        from tacorl_b200.networks.action_decoders.action_decoder_logistic import ActionDecoderLogistic
        self.action_decoder = ActionDecoderLogistic(state_dim=32, latent_plan_dim=16, hidden_size=64)
        self.perceptual_encoder = torch.nn.Linear(1, 1)
        self.actor = torch.nn.Linear(1, 1)
        self.action_decoder_modalities = ["rgb_static"]


@pytest.mark.parametrize("n_envs", [0, 65, -1, 2.0, True, "8"])
def test_policy_rejects_env_counts_outside_1_to_64(n_envs):
    from tacorl_b200.rollout import RolloutPolicy
    m = _Fake().eval()
    with pytest.raises(ValueError, match="n_envs"):
        RolloutPolicy(m, n_envs)


def test_policy_rejects_a_module_in_training_mode_or_without_a_decoder():
    from tacorl_b200.rollout import RolloutPolicy
    with pytest.raises(ValueError, match="eval"):
        RolloutPolicy(_Fake().train(), 4)
    with pytest.raises(ValueError, match="TACO-RL"):
        RolloutPolicy(torch.nn.Linear(2, 2).eval(), 4)


def test_policy_rejects_bad_env_ids():
    from tacorl_b200.rollout import RolloutPolicy
    m = _Fake().eval()
    for ids in ([0, 1, 2], [0, 1, 2, -1], [0, 1, 2, 2 ** 31]):
        with pytest.raises(ValueError, match="env_ids"):
            RolloutPolicy(m, 4, env_ids=ids)


def test_policy_on_a_cpu_module_has_no_fallback():
    from tacorl_b200 import _lib
    from tacorl_b200.rollout import RolloutPolicy
    with pytest.raises(_lib.TacorlLibraryError, match="CUDA"):
        RolloutPolicy(_Fake().eval(), 4)


def test_row_and_image_validation():
    from tacorl_b200.rollout import RolloutPolicy, _rows_list
    assert _rows_list(3, 8) == [3] and _rows_list([1, 5], 8) == [1, 5] and _rows_list(torch.tensor([0, 7]), 8) == [0, 7]
    for bad in ([8], [-1], [1, 1], [], [1.0], [True]):
        with pytest.raises(ValueError):
            _rows_list(bad, 8)
    p = object.__new__(RolloutPolicy)
    img = torch.zeros(2, 3, 84, 84, dtype=torch.uint8)
    p._check_images({"rgb_static": img}, ["rgb_static"], 2, "obs")
    for bad, msg in (({"rgb_gripper": img}, "modalities"), ({"rgb_static": img[:1]}, r"\(2, 3, H, W\)"),
                     ({"rgb_static": img[:, :2]}, r"\(2, 3, H, W\)"), ({"rgb_static": img.double()}, "uint8"),
                     ({"rgb_static": img, "rgb_gripper": img}, "modalities"), ([img], "dict")):
        with pytest.raises(ValueError, match=msg):
            p._check_images(bad, ["rgb_static"], 2, "obs")
