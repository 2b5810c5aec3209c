"""TEST INFRASTRUCTURE — CPU restatement of the rollout policy's PlayLMP and flat-CQL support and of its sampler
(tacorl_b200/rollout.py, tacorl_rollout_policy_sample in csrc/rollout.cu, DESIGN.md section 16.1): the policy's
counter-based uniforms, TanhNormal and GumbelSoftmax samples in fp64 from them, and RolloutOracle extended to PlayLMP,
flat CQL and sampled plans / actions.  Built from oracle.rollout_oracle and tacorl_oracle's reference restatements."""
import numpy as np
import torch

from oracle import replay_oracle as RO
from oracle import rollout_oracle as R
from oracle import tacorl_oracle as O
from oracle.rollout_oracle import decoder_step, sample, uniforms

POLICY_DRAW0 = 32                             # the policy sampler's first draw (the decoder's are 0..16)


def _u24(w):
    return torch.from_numpy((np.asarray(w) >> 8).astype(np.float32) * np.float32(2.0 ** -24))


def policy_uniforms(seed, t, env_id, A, gripper):
    """The policy sampler's uniforms of one step of one environment: continuous dimension d < A takes words 0 and 1 of
    the Philox4x32-10 draw j = 32 + d (key (lo32(seed), hi32(seed)), counter (lo32(t), hi32(t), env_id, j)) as u_a and
    u_b, (w >> 8) 2^-24; the gripper takes words 0 and 1 of draw 32 + A as u_0 and u_1.  t and env_id may be
    broadcastable integer arrays.  Returns (u_a (..., A), u_b (..., A), u_grip (..., 2) or None) float32 tensors."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    t = np.asarray(t, dtype=np.uint64)
    env = np.asarray(env_id, dtype=np.uint64)
    t, env = np.broadcast_arrays(t, env)
    draws = np.arange(POLICY_DRAW0, POLICY_DRAW0 + A + (1 if gripper else 0), dtype=np.uint64)
    w0, w1, _, _ = RO.philox4x32_10((t & np.uint64(0xFFFFFFFF))[..., None], (t >> np.uint64(32))[..., None],
                                    env[..., None], draws, seed & 0xFFFFFFFF, seed >> 32)
    ua, ub = _u24(w0), _u24(w1)
    grip = torch.stack([ua[..., A], ub[..., A]], -1) if gripper else None
    return ua[..., :A], ub[..., :A], grip


def tanh_normal_sample(mean, std, ua, ub):
    """TanhNormal.sample() from the uniforms, in fp64: tanh(mean + std sqrt(-2 ln(1 - u_a)) cos(2 pi u_b))."""
    ua, ub = ua.double(), ub.double()
    z = torch.sqrt(-2.0 * torch.log1p(-ua)) * torch.cos(2.0 * np.pi * ub)
    return torch.tanh(mean.double() + std.double() * z)


def gumbel_scores(logits, u):
    """GumbelSoftmax.sample()'s scores in fp64: normalised logits - log(-log(u)) (u = 0 scores -inf)."""
    norm = logits.double() - logits.double().logsumexp(dim=-1, keepdim=True)
    return norm - torch.log(-torch.log(u.double()))


def gripper_sample(logits, u):
    """2 argmax - 1 of gumbel_scores (ties -> class 0, torch.argmax's first maximum)."""
    return O.gumbel_argmax(logits.double(), u.double(), False).double() * 2.0 - 1.0


class RolloutOracle(R.RolloutOracle):
    """oracle.rollout_oracle.RolloutOracle for a TACO-RL (kind "tacorl"), PlayLMP ("play_lmp") or flat-CQL ("cql")
    module; deterministic=False samples the plans (TACO-RL, PlayLMP) or the actions (flat CQL) from policy_uniforms."""

    def __init__(self, P, n_envs, hidden, latent, kind="tacorl", deterministic=True, **kw):
        super().__init__(P, n_envs, hidden, latent, **kw)
        self.kind, self.deterministic = kind, deterministic

    def _policy_input(self, o, r):
        """cat(encoder(obs), goal_encoder(encoder(goal))) of the high-level policy (actor / plan proposal)."""
        if self.kind == "play_lmp":
            enc = lambda x, m: O.lmp_encoder(self.P, f"perceptual_encoder.networks.{m}.", x)
            e = torch.cat([enc(o[m], m) for m in self.obs_mods], -1)
            g = torch.cat([enc(self.goal[r][m], m) for m in self.goal_mods], -1)
            return torch.cat([e, O.goal_encoder(self.P, "goal_encoder.", g)], -1)
        return O.visual_emb(self.P, "actor.", o, self.goal[r], self.obs_mods, self.goal_mods)

    def step(self, obs):
        """obs: {modality: (n, 3, H, W)} -> (actions (n, 7), logits (n, 182), or None for flat CQL)."""
        acts, logits = [], []
        for r in range(self.n):
            o = {m: obs[m][r:r + 1].to(self.dtype) for m in obs}
            if self.kind == "cql":
                mu, std, lg = O.mlp_policy_gripper(self.P, "actor.actor.policy.", self._policy_input(o, r))
                if self.deterministic:     # Actor.get_actions(deterministic=True)
                    grip = torch.argmax(torch.softmax(lg, -1), -1).to(self.dtype) * 2.0 - 1
                    acts.append(torch.cat([torch.tanh(mu)[0], grip]))
                else:
                    ua, ub, ug = policy_uniforms(self.seed, self.t[r], self.env_ids[r], mu.shape[-1], True)
                    acts.append(torch.cat([tanh_normal_sample(mu[0], std[0], ua, ub),
                                           gripper_sample(lg[0], ug)[None]]).to(self.dtype))
                self.t[r] += 1
                continue
            if self.pending[r]:
                pre = "plan_proposal.policy." if self.kind == "play_lmp" else "actor.actor.policy."
                mu, std = O.mlp_policy(self.P, pre, self._policy_input(o, r))
                if self.deterministic:
                    self.plan[r] = torch.tanh(mu)[0]
                else:           # drawn at the t of the row's next decoder step, from draws 32 + d
                    ua, ub, _ = policy_uniforms(self.seed, self.t[r], self.env_ids[r], mu.shape[-1], False)
                    self.plan[r] = tanh_normal_sample(mu[0], std[0], ua, ub).to(self.dtype)
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
        return torch.stack(acts), (torch.stack(logits) if logits else None)
