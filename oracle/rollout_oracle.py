"""TEST INFRASTRUCTURE — CPU restatement of the batched rollout policy (tacorl_b200/rollout.py, csrc/rollout.cu,
DESIGN.md section 16): the counter-based sampling uniforms and per-environment stepping of plan, hidden state and
action, built from tacorl_oracle's reference restatements.  The product package never imports this module."""
import numpy as np
import torch

from oracle import replay_oracle as RO
from oracle import tacorl_oracle as O

N_DIMS, N_MIX = 6, 10
N_UNIFORMS = N_DIMS * N_MIX + N_DIMS          # 60 Gumbel uniforms u1, then 6 logistic uniforms u2


def uniforms(seed, t, env_id):
    """The 66 uniforms of one control step of one environment: uniform i is word i mod 4 of the Philox4x32-10 draw with
    key (lo32(seed), hi32(seed)) and counter (lo32(t), hi32(t), env_id, i div 4), as (w >> 8) 2^-24.  t and env_id may be
    broadcastable integer arrays.  Returns (u1 (..., 6, 10), u2 (..., 6)) float32 tensors: u1[d][k] is uniform 10 d + k,
    u2[d] is uniform 60 + d."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    t = np.asarray(t, dtype=np.uint64)
    env = np.asarray(env_id, dtype=np.uint64)
    t, env = np.broadcast_arrays(t, env)
    draws = np.arange((N_UNIFORMS + 3) // 4, dtype=np.uint64)
    words = RO.philox4x32_10((t & np.uint64(0xFFFFFFFF))[..., None], (t >> np.uint64(32))[..., None], env[..., None],
                             draws, seed & 0xFFFFFFFF, seed >> 32)
    w = np.stack(words, -1).reshape(*t.shape, -1)[..., :N_UNIFORMS]          # uniform i = word i % 4 of draw i // 4
    u = torch.from_numpy((w >> 8).astype(np.float32) * np.float32(2.0 ** -24))
    return u[..., :N_DIMS * N_MIX].reshape(*t.shape, N_DIMS, N_MIX), u[..., N_DIMS * N_MIX:]


def decoder_step(P, plan, emb, h, pre="action_decoder."):
    """One step of ActionDecoderLogistic.forward with h0 = h (2, B, H): returns ((probs, log_scales, means, grip) each
    (B, ...), h_n)."""
    lp, ls, mm, grip, hn = O.action_decoder_forward(P, pre, plan, emb.unsqueeze(1), h0=h)
    return (lp[:, 0], ls[:, 0], mm[:, 0], grip[:, 0]), hn


def sample(heads, u1, u2, gripper_bounds=(-1.0, 1.0)):
    """dlm_sample of one step: heads from decoder_step, u1 (B, 6, 10), u2 (B, 6) -> actions (B, 7)."""
    lp, ls, mm, grip = heads
    return O.dlm_sample(lp[:, None], ls[:, None], mm[:, None], grip[:, None], u1[:, None], u2[:, None],
                        gripper_bounds)[:, 0]


class RolloutOracle:
    """RolloutPolicy on the CPU, one environment at a time.  P: parameter dict (tacorl_oracle.params_from) of a TACO-RL
    module; images are normalised float tensors."""

    def __init__(self, P, n_envs, hidden, latent, seed=0, env_ids=None, obs_mods=("rgb_static",),
                 goal_mods=("rgb_static",), dec_mods=None, dtype=torch.float64):
        self.P, self.n, self.seed, self.dtype = P, n_envs, seed, dtype
        self.env_ids = list(range(n_envs)) if env_ids is None else list(env_ids)
        self.obs_mods, self.goal_mods = tuple(obs_mods), tuple(goal_mods)
        self.dec_mods = tuple(dec_mods if dec_mods is not None else obs_mods)
        self.plan = torch.zeros(n_envs, latent, dtype=dtype)
        self.h = torch.zeros(2, n_envs, hidden, dtype=dtype)
        self.t = [0] * n_envs
        self.goal = [None] * n_envs
        self.pending = [False] * n_envs

    def reset(self, rows, goal):
        self.set_goal(rows, goal)
        for r in rows:
            self.t[r] = 0

    def set_goal(self, rows, goal):
        for i, r in enumerate(rows):
            self.goal[r] = {m: goal[m][i:i + 1].to(self.dtype) for m in self.goal_mods}
            self.pending[r] = True

    def replan(self, rows):
        for r in rows:
            self.pending[r] = True

    def step(self, obs):
        """obs: {modality: (n, 3, H, W)} -> (actions (n, 7), logits (n, 182))."""
        acts, logits = [], []
        for r in range(self.n):
            o = {m: obs[m][r:r + 1].to(self.dtype) for m in obs}
            if self.pending[r]:
                a_emb = O.visual_emb(self.P, "actor.", o, self.goal[r], self.obs_mods, self.goal_mods)
                mu, _ = O.mlp_policy(self.P, "actor.actor.policy.", a_emb)
                self.plan[r] = torch.tanh(mu)[0]
                self.h[:, r] = 0
                self.pending[r] = False
            emb = torch.cat([O.lmp_encoder(self.P, f"perceptual_encoder.networks.{m}.", o[m]) for m in self.dec_mods], -1)
            heads, hn = decoder_step(self.P, self.plan[r:r + 1], emb, self.h[:, r:r + 1])
            self.h[:, r:r + 1] = hn
            u1, u2 = uniforms(self.seed, self.t[r], self.env_ids[r])
            acts.append(sample(heads, u1[None].to(self.dtype), u2[None].to(self.dtype))[0])
            lp, ls, mm, grip = heads
            logits.append(torch.cat([lp.reshape(-1), mm.reshape(-1), ls.reshape(-1), grip.reshape(-1)]))
            self.t[r] += 1
        return torch.stack(acts), torch.stack(logits)
