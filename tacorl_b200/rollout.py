"""Batched rollout policy of a trained TACO-RL, PlayLMP or flat-CQL agent: many environments, one CUDA-graph replay
per control step.

The reference's policy entry is single-environment and stateful (rollout_manager.py:364-386): a deterministic latent
plan from the visual actor, `clear_hidden_state()`, then one `act()` per control step, with ONE hidden state and one
`torch.rand` draw for the whole batch.  `RolloutPolicy` keeps per-environment plans, hidden states, goals and step
counters on the device, so environments reset, change subtask and replan independently, and draws each environment's
sampling noise from its own counter (Philox4x32-10 keyed by the seed, counter = (step, env_id, draw)): an
environment's noise depends only on the seed, its env_id and its own step count, never on which other environments
share the batch, and the decoder step is batch-invariant.  DESIGN.md section 16 states the rules.

    policy = RolloutPolicy(module, n_envs, seed=0)
    policy.reset(rows, goal)        # goal images of these environments; their step counters restart at 0
    actions = policy.step(obs)      # {modality: (n_envs, 3, H, W)} uint8 or normalised fp32 -> (n_envs, 7)

The decoder step is `tacorl_rollout_decoder_step` and sampled plans and flat-CQL actions are drawn by
`tacorl_rollout_policy_sample` (csrc/rollout.cu); the encoders and the actor run through the same library kernels as
training.  Nothing here changes the module: `act()`, `clear_hidden_state()` and training are untouched.

A TACO-RL policy built with `plan_search=PlanSearch(...)` replans by a cross-entropy-method search over the latent plan
scored by the module's twin critics (`tacorl_plan_search_*`, csrc/plan_search.cu, DESIGN.md section 16.2) instead of
taking the actor's tanh(mean); `policy.plan_value` holds min(Q1, Q2) of each row's current plan."""
import ctypes

import numpy as np
import torch

from . import _lib as L
from . import ops

MAX_ENVS = 64


def _rows_list(rows, n):
    if torch.is_tensor(rows):
        rows = rows.detach().cpu().reshape(-1).tolist()
    elif isinstance(rows, (int, np.integer)):
        rows = [rows]
    out = []
    for r in rows:
        if isinstance(r, (bool, np.bool_)) or not isinstance(r, (int, np.integer)):
            raise ValueError(f"rows must be integers, got {r!r}")
        if not 0 <= int(r) < n:
            raise ValueError(f"row {int(r)} out of range for {n} environments")
        out.append(int(r))
    if not out:
        raise ValueError("no rows given")
    if len(set(out)) != len(out):
        raise ValueError(f"duplicate rows {out}")
    return out


def decoder_weights(decoder):
    """The 16 fp32 tensors of tacorl_rollout_decoder_step, in the order of include/tacorl_b200.h."""
    rnn = decoder.rnn
    w = [getattr(rnn, f"{k}_l{l}") for l in range(2) for k in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
    for fc in (decoder.prob_fc, decoder.mean_fc, decoder.log_scale_fc, decoder.gripper_fc):
        w += [fc.weight, fc.bias]
    return [t.detach() for t in w]


def decoder_step(decoder, plan, emb, hidden, restart, seed, env_id, t, actions, logits=None, ws=None):
    """One control step of `decoder` (an ActionDecoderLogistic) for n = plan.shape[0] environments, in the current
    precision mode: hidden (2, n, H) and t (n, int64) are updated in place, actions (n, 7) and logits (n, 182, optional)
    are written.  ws: a zero-filled uint8 buffer of tacorl_rollout_ws_bytes(n, H) bytes kept between calls (a fresh one
    is allocated when None)."""
    n, P = plan.shape
    E, H = emb.shape[1], hidden.shape[2]
    w = decoder_weights(decoder)
    for x in w:
        if not x.is_contiguous():
            raise ValueError("decoder weights must be contiguous")
    shadows = [ops.shadow_of(w[i]) for i in (0, 1, 4, 5, 8, 10, 12, 14)]
    if ws is None:
        ws = torch.zeros(int(L.query("tacorl_rollout_ws_bytes", n, H)), dtype=torch.uint8, device=plan.device)
    L.call("tacorl_rollout_decoder_step", n, P, E, H, L.ptr(plan), L.ptr(emb), L.ptr(hidden), L.ptr_any(restart),
           L.ptr_array(w), L.ptr_array(shadows), ctypes.c_ulonglong(int(seed) & 0xFFFFFFFFFFFFFFFF), L.ptr_any(env_id),
           L.ptr_any(t), float(decoder._grip[0]), float(decoder._grip[1]), L.ptr(actions), L.ptr(logits),
           ctypes.c_void_p(ws.data_ptr()), ws.numel(), ops._STATE["prec"], L.stream())
    return actions


def policy_sample(mean, std, logits, mask, seed, env_id, t, out, advance_t=False):
    """Sample n = mean.shape[0] rows of a TanhNormal(mean, std) (n, A) arm, plus a GumbelSoftmax gripper when logits
    (n, 2) are given, from each row's counter-based noise (Philox draws 32 + d, DESIGN.md section 16), into out (n, >= A
    [+ 1]): tanh(mean + std z) and the gripper as 2 class - 1.  mask: None or (n,) int32, rows whose mask is 0 are not
    written.  advance_t: t (n, int64) is incremented after sampling.  fp32 in both precision modes."""
    n, A = mean.shape
    if std.shape != mean.shape or (logits is not None and logits.shape != (n, 2)):
        raise ValueError(f"policy_sample: mean {tuple(mean.shape)}, std {tuple(std.shape)}, logits "
                         f"{None if logits is None else tuple(logits.shape)}")
    if out.dim() != 2 or out.shape[0] != n or out.stride(1) != 1:
        raise ValueError(f"policy_sample: out must be ({n}, >= {A}) with unit column stride")
    if env_id.dtype != torch.int32 or t.dtype != torch.int64 or (mask is not None and mask.dtype != torch.int32):
        raise ValueError("policy_sample: env_id and mask are int32, t is int64")
    L.call("tacorl_rollout_policy_sample", n, A, L.ptr(mean.contiguous()), L.ptr(std.contiguous()),
           L.ptr(None if logits is None else logits.contiguous()), L.ptr_any(mask),
           ctypes.c_ulonglong(int(seed) & 0xFFFFFFFFFFFFFFFF), L.ptr_any(env_id), L.ptr_any(t), int(bool(advance_t)),
           L.ptr(out), out.stride(0), L.stream())
    return out


class PlanSearch:
    """Settings of the critic-guided plan search (DESIGN.md section 16.2): `iterations` rounds of `samples` candidate
    pre-tanh plans per replanning environment, drawn from a diagonal Gaussian that starts at the actor's head and is
    refitted to the `elites` best candidates by min(Q1, Q2), its std floored at `min_std`.  The plan is tanh of the
    best candidate of all rounds; candidate 0 of round 0 is the actor's deterministic plan."""

    def __init__(self, samples=128, elites=16, iterations=3, min_std=1e-3):
        for name, v in (("samples", samples), ("elites", elites), ("iterations", iterations)):
            if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, np.integer)):
                raise ValueError(f"PlanSearch: {name} must be an integer (got {v!r})")
        samples, elites, iterations = int(samples), int(elites), int(iterations)
        if not 32 <= samples <= 512 or samples % 32:
            raise ValueError(f"PlanSearch: samples must be a multiple of 32 in 32..512 (got {samples})")
        if not 1 <= elites <= samples:
            raise ValueError(f"PlanSearch: elites must be in 1..samples = {samples} (got {elites})")
        if not 1 <= iterations <= 8:
            raise ValueError(f"PlanSearch: iterations must be in 1..8 (got {iterations})")
        if (isinstance(min_std, (bool, np.bool_)) or not isinstance(min_std, (int, float, np.integer, np.floating))
                or not np.isfinite(min_std) or not np.float32(min_std) > 0):
            raise ValueError(f"PlanSearch: min_std must be a finite number > 0 (got {min_std!r})")
        self.samples, self.elites, self.iterations, self.min_std = samples, elites, iterations, float(min_std)

    def __repr__(self):
        return (f"PlanSearch(samples={self.samples}, elites={self.elites}, iterations={self.iterations}, "
                f"min_std={self.min_std})")


def critic_layers(qnet):
    """The fp32 (W, b) pairs of an MLPQNetwork: its SiLU layers, then the output layer (W (1, H), b (1))."""
    if not hasattr(qnet, "fc_layers") or not hasattr(qnet, "out"):
        raise ValueError("the plan search scores plans with MLPQNetwork critics")
    layers = [(fc.weight.detach(), fc.bias.detach()) for fc in qnet.fc_layers] + [(qnet.out.weight.detach(),
                                                                                   qnet.out.bias.detach())]
    H = layers[0][0].shape[0]
    for W, b in layers[1:-1]:
        if W.shape != (H, H):
            raise ValueError(f"the plan search needs equal hidden widths (got {tuple(W.shape)} after width {H})")
    if layers[-1][0].shape != (1, H):
        raise ValueError("the critic's output layer must be Linear(hidden, 1)")
    for W, b in layers:
        if not (W.is_contiguous() and b.is_contiguous()):
            raise ValueError("critic weights must be contiguous")
    return layers


class SearchBuffers:
    """Device buffers of a plan search over n environments and K samples: the workspace of tacorl_plan_search_*, the
    candidates z (n K, P) and their scores (n, K) of the latest round, the refitted (mu, sigma) (n, P) and the best
    candidate so far, best_z (n, P) and best_s (n)."""

    def __init__(self, n, K, P, H, device):
        f32 = dict(device=device, dtype=torch.float32)
        self.n, self.K, self.P, self.H = n, K, P, H
        self.ws = torch.empty(int(L.query("tacorl_plan_search_ws_bytes", n, K, P, H)), dtype=torch.uint8, device=device)
        self.z = torch.empty(n * K, P, **f32)
        self.scores = torch.empty(n, K, **f32)
        self.mu, self.sigma, self.best_z = (torch.empty(n, P, **f32) for _ in range(3))
        self.best_s = torch.empty(n, **f32)


def plan_search(critics, eo, eg, mean, std, search, seed, env_id, t, restart, plan, plan_value, bufs, trace=None,
                uniforms=None):
    """The critic-guided plan search of n = mean.shape[0] environments in the current precision mode (DESIGN.md
    section 16.2).  critics: the two MLPQNetworks; eo / eg: per critic its (n, Do) observation and (n, Dg) goal
    embeddings; mean, std (n, P): the actor's head (ops.gauss_head); restart: None or (n,) int32, rows whose flag is 0
    keep their plan (n, P) and plan_value (n,).  bufs: SearchBuffers(n, K, P, H).  trace: None or a list that receives,
    after every round, copies of that round's candidates, scores, refit and best-so-far (tests; not graph-capturable).
    uniforms: None or a list that receives each round's (n K, P, 2) Philox uniforms (tests)."""
    n, P = mean.shape
    K, E, I = search.samples, search.elites, search.iterations
    q = [critic_layers(c) for c in critics]
    H, nl = q[0][0][0].shape[0], len(q[0]) - 1
    if len(q[1]) != len(q[0]) or q[1][0][0].shape != q[0][0][0].shape:
        raise ValueError("the two critics must have the same shapes")
    Do, Dg = eo[0].shape[1], eg[0].shape[1]
    for j in range(2):
        if eo[j].shape != (n, Do) or eg[j].shape != (n, Dg) or q[j][0][0].shape[1] != Do + Dg + P:
            raise ValueError(f"plan_search: critic {j + 1} takes {q[j][0][0].shape[1]} inputs, embeddings "
                             f"{tuple(eo[j].shape)} + {tuple(eg[j].shape)} + plan {P}")
    if (bufs.n, bufs.K, bufs.P, bufs.H) != (n, K, P, H):
        raise ValueError("plan_search: buffers of another shape")
    if env_id.dtype != torch.int32 or t.dtype != torch.int64 or (restart is not None and restart.dtype != torch.int32):
        raise ValueError("plan_search: env_id and restart are int32, t is int64")
    eo = [x.contiguous() for x in eo]
    eg = [x.contiguous() for x in eg]
    mean, std = mean.contiguous(), std.contiguous()
    prec = ops._STATE["prec"]
    sd = ctypes.c_ulonglong(int(seed) & 0xFFFFFFFFFFFFFFFF)
    ws = ctypes.c_void_p(bufs.ws.data_ptr())
    (W1, b1), (W2, b2) = q[0][-1], q[1][-1]
    for k in range(I):
        mu, sg = (mean, std) if k == 0 else (bufs.mu, bufs.sigma)
        u = torch.empty(n * K, P, 2, device=mean.device) if uniforms is not None else None
        L.call("tacorl_plan_search_sample_l0", n, K, P, Do, Dg, H, k, L.ptr(mu), L.ptr(sg),
               L.ptr(eo[0]), L.ptr(eg[0]), L.ptr(q[0][0][0]), L.ptr(q[0][0][1]),
               L.ptr(eo[1]), L.ptr(eg[1]), L.ptr(q[1][0][0]), L.ptr(q[1][0][1]),
               sd, L.ptr_any(env_id), L.ptr_any(t), L.ptr(bufs.z), L.ptr(u), ws, bufs.ws.numel(), prec, L.stream())
        for l in range(1, nl):
            (Wa, ba), (Wb, bb) = q[0][l], q[1][l]
            L.call("tacorl_plan_search_hidden", n, K, H, l, L.ptr(Wa), L.ptr_any(ops.shadow_of(Wa)), L.ptr(ba),
                   L.ptr(Wb), L.ptr_any(ops.shadow_of(Wb)), L.ptr(bb), ws, bufs.ws.numel(), prec, L.stream())
        L.call("tacorl_plan_search_select", n, K, P, H, nl, E, k, int(k == I - 1), float(search.min_std),
               L.ptr(bufs.z), L.ptr(W1), L.ptr(b1), L.ptr(W2), L.ptr(b2), L.ptr(bufs.scores), L.ptr(bufs.mu),
               L.ptr(bufs.sigma), L.ptr(bufs.best_z), L.ptr(bufs.best_s), L.ptr_any(restart), L.ptr(plan),
               L.ptr(plan_value), ws, bufs.ws.numel(), L.stream())
        if uniforms is not None:
            uniforms.append(u)
        if trace is not None:
            trace.append({k2: getattr(bufs, k2).clone() for k2 in ("z", "scores", "mu", "sigma", "best_z", "best_s")})
    return plan


def _module_kind(module):
    """"play_lmp", "cql" (flat CQL: a CQL_Offline without an action decoder) or "tacorl" (everything else, checked as
    a TACO-RL module)."""
    from .modules.cql.cql_offline_lightning import CQL_Offline
    from .modules.play_lmp.play_lmp_for_rl import PlayLMP
    if isinstance(module, PlayLMP):
        return "play_lmp"
    if isinstance(module, CQL_Offline) and not hasattr(module, "action_decoder"):
        return "cql"
    return "tacorl"


def _check_decoder(dec):
    if not hasattr(dec, "_grip") or getattr(dec.rnn, "num_layers", None) != 2 or dec.rnn.bidirectional:
        raise ValueError("RolloutPolicy covers the two-layer ActionDecoderLogistic")


def _cat(ts):
    return ts[0] if len(ts) == 1 else torch.cat(ts, dim=-1)


class RolloutPolicy:
    """Batched rollout of a TACO-RL, PlayLMP or flat-CQL module (eval mode, on its CUDA device) for 1..64 environments.

    reset(rows, goal)    new episode: goal images for these rows, step counter 0, replan at their next step
    set_goal(rows, goal) next subtask: new goal, replan at the next step, step counter kept
    replan(rows)         new plan and zero hidden state at the next step (every plan_duration steps; not flat CQL)
    step(obs)            one control step of every environment -> (n_envs, 7) actions

    TACO-RL and PlayLMP: a replanning row takes a plan from the high-level policy (TACO-RL's actor, PlayLMP's
    plan_proposal) on its encoder embedding of the current observation and the goal embedding
    goal_encoder(encoder(goal)) (computed once, at reset / set_goal): tanh(mean) with deterministic=True (the
    reference's deterministic actor call), a TanhNormal sample drawn from the row's own noise otherwise (PlayLMP's
    `pp_dist.sample()`).  Its hidden state restarts at zero and its first decoder step uses the same frame.  The decoder
    consumes perceptual_encoder.get_state_from_observation(obs, action_decoder_modalities), as `act()` does; PlayLMP's
    plan proposal reads the same encoder, so each modality is encoded once per step.
    Flat CQL: every step is the actor on cat(encoder(obs), goal embedding): Actor.get_actions(deterministic=True)
    (tanh(mean), argmax gripper), or with deterministic=False a TanhNormal arm and GumbelSoftmax gripper sample.
    plan_search=PlanSearch(...) (TACO-RL, deterministic=True only): a replanning row's plan comes from a cross-entropy
    search scored by min(Q1, Q2) of the module's critics, started at the actor's head (DESIGN.md section 16.2);
    reset / set_goal also cache each critic's goal embedding, the replan step adds one pass of each critic's encoder,
    and `plan_value` (n,) holds each row's min(Q1, Q2) of its current plan (NaN before its first replan).

    Each step is one CUDA-graph replay of one of two graphs, with and without a replan (the replan graph runs the actor
    for every row and keeps the plan of the flagged rows only; flat CQL has one graph); the host picks it from its own
    bookkeeping.  `step`
    copies the observation into `static_obs`; a caller may instead write there and call `step()` with no argument.
    The returned actions tensor is the policy's output buffer: it is overwritten by the next step.  The policy reads the
    module's live parameters: an optimiser step, `load_state_dict` or a torch-side edit between steps is seen by the
    next step, and a step whose parameters or bf16 shadows moved since the capture (an optimiser built or dropped
    since) captures its graphs again."""

    def __init__(self, module, n_envs, seed=0, env_ids=None, use_graphs=True, deterministic=True, plan_search=None):
        kind = _module_kind(module)
        if plan_search is not None:
            if not isinstance(plan_search, PlanSearch):
                raise ValueError(f"plan_search must be a PlanSearch or None (got {type(plan_search).__name__})")
            if kind != "tacorl" or not all(hasattr(module, a) for a in ("q1", "q2", "actor")):
                raise ValueError("the plan search needs a TACO-RL module: PlayLMP has no critic and flat CQL no plan")
            if deterministic is not True:
                raise ValueError("the plan search replaces the actor's plan: it cannot be combined with "
                                 "deterministic=False")
        if kind == "tacorl":
            for attr in ("actor", "action_decoder", "perceptual_encoder", "action_decoder_modalities"):
                if not hasattr(module, attr):
                    raise ValueError(f"RolloutPolicy needs a TACO-RL, PlayLMP or flat-CQL module (no `{attr}`)")
            _check_decoder(module.action_decoder)
        elif kind == "play_lmp":
            _check_decoder(module.action_decoder)
            if not hasattr(module.plan_proposal, "policy") or module.plan_proposal.discrete_gripper:
                raise ValueError("RolloutPolicy covers a PlayLMP whose plan proposal is a continuous Actor")
        elif not module.actor.discrete_gripper:
            raise ValueError("RolloutPolicy covers flat CQL with a discrete (GumbelSoftmax) gripper")
        if not isinstance(deterministic, bool):
            raise ValueError(f"deterministic must be a bool (got {deterministic!r})")
        if isinstance(n_envs, bool) or not isinstance(n_envs, (int, np.integer)) or not 1 <= int(n_envs) <= MAX_ENVS:
            raise ValueError(f"n_envs must be an integer in 1..{MAX_ENVS} (got {n_envs!r}); build several policies for more")
        if module.training:
            raise ValueError("put the module in eval mode (module.eval()) before building a RolloutPolicy")
        n = int(n_envs)
        if env_ids is None:
            env_ids = list(range(n))
        env_ids = [int(e) for e in (env_ids.tolist() if torch.is_tensor(env_ids) else env_ids)]
        if len(env_ids) != n or any(not 0 <= e < 2 ** 31 for e in env_ids):
            raise ValueError(f"env_ids must be {n} integers in [0, 2^31)")
        dev = next(module.parameters()).device
        if dev.type != "cuda":
            raise L.TacorlLibraryError("RolloutPolicy runs on a CUDA device (there is no CPU path)")
        self.module, self.n, self.seed, self.device = module, n, int(seed), dev
        self.kind, self.deterministic = kind, deterministic
        self.search = plan_search
        self.use_graphs = bool(use_graphs)
        # what the step reads: the encoder of the actor's (plan proposal's) input, its goal encoder and policy, and the
        # decoder with its encoder (None for flat CQL)
        if kind == "play_lmp":
            self._enc, self._goal_enc, self._net = module.perceptual_encoder, module.goal_encoder, module.plan_proposal
            self.env_mods = list(module.plan_proposal_obs_modalities)
            self.goal_mods = list(module.plan_proposal_goal_modalities)
            nets = (module.perceptual_encoder, module.goal_encoder, module.plan_proposal, module.action_decoder)
        else:
            actor = module.actor
            self._enc, self._goal_enc, self._net = actor.encoder, actor.goal_encoder, actor.actor
            self.env_mods, self.goal_mods = list(actor.env_modalities), list(actor.goal_modalities)
            nets = ((module.perceptual_encoder, actor, module.action_decoder) if kind == "tacorl"
                    else tuple(m for m in (actor.encoder, actor.goal_encoder, actor.actor) if m is not None))
        self._dec = None if kind == "cql" else module.action_decoder
        self.dec_mods = [] if kind == "cql" else list(module.action_decoder_modalities)
        self.obs_mods = list(dict.fromkeys(self.dec_mods + self.env_mods))
        f32 = dict(device=dev, dtype=torch.float32)
        if self._dec is not None:
            dec = self._dec
            self.P = dec.latent_plan_dim
            self.H = dec.rnn.hidden_size
            self.E = dec.rnn.input_size - self.P
            if self.P % 4 or self.E % 4 or self.H % 8:
                raise ValueError(f"decoder sizes plan {self.P} / embedding {self.E} / hidden {self.H} are not supported")
            self.plan = torch.zeros(n, self.P, **f32)
            self.hidden = torch.zeros(2, n, self.H, **f32)
            self.logits = torch.zeros(n, 182, **f32)
            self.ws = torch.zeros(int(L.query("tacorl_rollout_ws_bytes", n, self.H)), dtype=torch.uint8, device=dev)
        else:
            self.plan = self.hidden = None
        self.goal_emb = torch.zeros(n, self._net.goal_dim, **f32)
        self.restart = torch.zeros(n, device=dev, dtype=torch.int32)
        self.env_id = torch.tensor(env_ids, device=dev, dtype=torch.int32)
        self.t = torch.zeros(n, device=dev, dtype=torch.int64)
        self.actions = torch.zeros(n, 7, **f32)
        self.static_obs = None
        self._replan = np.zeros(n, dtype=np.int32)
        self._has_goal = np.zeros(n, dtype=bool)
        self._graphs = {}
        self._pool = None
        self.launches = {}            # (replan, precision) -> library launches recorded in that graph
        self.plan_value = None
        self._critics = []
        if plan_search is not None:
            self._critics = [module.q1, module.q2]
            for q in self._critics:
                critic_layers(q.critic.Q)
                if not set(q.env_modalities) <= set(self.obs_mods) or not set(q.goal_modalities) <= set(self.goal_mods):
                    raise ValueError("the critics must read the actor's observation and goal modalities")
            H = module.q1.critic.Q.fc_layers[0].weight.shape[0]
            if self.P > 64 or H % 32 or not 32 <= H <= 1024:
                raise ValueError(f"the plan search covers plans of <= 64 dimensions and critic widths that are "
                                 f"multiples of 32 in 32..1024 (plan {self.P}, critic {H})")
            self.plan_value = torch.full((n,), float("nan"), **f32)
            self.q_goal_emb = [None, None]
            self._search_bufs = SearchBuffers(n, plan_search.samples, self.P, H, dev)
            nets = nets + (module.q1, module.q2)
        self._tensors = [x for mod in nets for x in list(mod.parameters()) + list(mod.buffers())]
        self.captures = 0

    # ------------------------------------------------------------------------------------------------ validation
    def _check_images(self, imgs, mods, rows, what):
        if not isinstance(imgs, dict) or set(imgs) != set(mods):
            got = sorted(imgs) if isinstance(imgs, dict) else type(imgs).__name__
            raise ValueError(f"{what} must be a dict with the modalities {sorted(mods)} (got {got})")
        for m in mods:
            x = imgs[m]
            if not torch.is_tensor(x) or x.dim() != 4 or x.shape[0] != rows or x.shape[1] != 3:
                shape = tuple(x.shape) if torch.is_tensor(x) else type(x).__name__
                raise ValueError(f"{what}[{m!r}] must be ({rows}, 3, H, W), got {shape}")
            if x.dtype not in (torch.uint8, torch.float32):
                raise ValueError(f"{what}[{m!r}] must be uint8 frames or normalised float32, got {x.dtype}")

    # ------------------------------------------------------------------------------------------------ episode control
    @torch.no_grad()
    def _set_goal(self, rows, goal):
        rows = _rows_list(rows, self.n)
        self._check_images(goal, self.goal_mods, len(rows), "goal")
        g = {m: goal[m].to(self.device) for m in self.goal_mods}
        emb = self._enc.get_state_from_observation(observation=g, modalities=self.goal_mods).reshape(len(rows), -1)
        if self._goal_enc is not None:
            emb = self._goal_enc(emb)
        self.goal_emb[rows] = emb.reshape(len(rows), -1)
        for j, q in enumerate(self._critics):        # goal_encoder_qj(encoder_qj(goal)), the critics' goal embedding
            ge = q.encoder.get_state_from_observation(observation=g, modalities=q.goal_modalities).reshape(len(rows), -1)
            if q.goal_encoder is not None:
                ge = q.goal_encoder(ge)
            ge = ge.reshape(len(rows), -1)
            if self.q_goal_emb[j] is None:
                self.q_goal_emb[j] = torch.zeros(self.n, ge.shape[1], device=self.device, dtype=torch.float32)
            self.q_goal_emb[j][rows] = ge
        self._has_goal[rows] = True
        if self._dec is not None:
            self._replan[rows] = 1
        return rows

    def reset(self, rows, goal):
        """New episode for `rows`: goal images, step counter 0, replan (plan + zero hidden state) at the next step."""
        rows = self._set_goal(rows, goal)
        self.t[rows] = 0

    def set_goal(self, rows, goal):
        """Next subtask for `rows`: new goal, replan at the next step; the step counter keeps counting."""
        self._set_goal(rows, goal)

    def replan(self, rows):
        """New plan and zero hidden state for `rows` at the next step."""
        if self._dec is None:
            raise ValueError("flat CQL has no plan: every step already runs the actor")
        rows = _rows_list(rows, self.n)
        self._replan[rows] = 1

    # ------------------------------------------------------------------------------------------------ stepping
    def _embed(self, enc, mods):
        return enc.get_state_from_observation(observation=self.static_obs, modalities=mods).reshape(self.n, -1)

    def _run(self, replan):
        """The work of one step on the static buffers (what a graph captures)."""
        with torch.no_grad():
            if self._dec is None:
                self._act(self._embed(self._enc, self.env_mods))
                return
            if self.kind == "play_lmp":       # plan proposal and decoder read the same encoder: each view once
                per = self._enc.get_state_from_observation(observation=self.static_obs, modalities=self.obs_mods,
                                                           cat_output=False)
                per = {k: v.reshape(self.n, -1) for k, v in per.items()}
                emb = _cat([per[k] for k in self.dec_mods])
                e = _cat([per[k] for k in self.env_mods]) if replan else None
            else:
                emb = self._embed(self.module.perceptual_encoder, self.dec_mods)
                e = self._embed(self._enc, self.env_mods) if replan else None
            if replan:
                out = self._net(e, self.goal_emb)
                if self.search is not None:     # the flagged rows' plans and values from the critic-guided search
                    eo = [self._embed(q.encoder, q.env_modalities) for q in self._critics]
                    plan_search([q.critic.Q for q in self._critics], eo, self.q_goal_emb, out[0], out[1], self.search,
                                self.seed, self.env_id, self.t, self.restart, self.plan, self.plan_value,
                                self._search_bufs)
                elif self.deterministic:
                    new_plan = torch.tanh(out[0])
                    self.plan.copy_(torch.where(self.restart.unsqueeze(1) != 0, new_plan, self.plan))
                else:         # the flagged rows' plans, drawn at the t their first decoder step reads
                    policy_sample(out[0], out[1], None, self.restart, self.seed, self.env_id, self.t, self.plan)
            decoder_step(self._dec, self.plan, emb.contiguous(), self.hidden, self.restart, self.seed,
                         self.env_id, self.t, self.actions, self.logits, self.ws)

    def _act(self, e):
        """Flat CQL: the actor on cat(e, goal embedding) -> actions, then t += 1."""
        mean, std, logits = self._net(e, self.goal_emb)
        if self.deterministic:            # Actor.get_actions(deterministic=True)
            A = mean.shape[1]
            self.actions[:, :A].copy_(torch.tanh(mean))
            grip = torch.argmax(torch.softmax(logits, dim=-1), dim=-1).to(torch.float32) * 2.0 - 1
            self.actions[:, A].copy_(grip)
            self.t.add_(1)
        else:
            policy_sample(mean, std, logits, None, self.seed, self.env_id, self.t, self.actions, advance_t=True)

    def _signature(self):
        """What decides the device addresses a captured step reads.  A graph bakes them in: an optimiser built later
        moves the parameters into its flat buffer, and a dropped optimiser takes its bf16 shadows with it, so a step
        whose signature differs from its graph's captures again.  The parameters' and buffers' addresses, the live
        optimisers' shadow buffers (a parameter's shadow is its owner's buffer at the parameter's offset) and the cached
        shadows of frozen parameters determine every address `ops.shadow_of` can hand the kernels."""
        return (ops.get_precision(), tuple(x.data_ptr() for x in self._tensors),
                frozenset((id(o), o.shadow.data_ptr()) for o in ops._SHADOW_OWNERS),
                frozenset(id(v[2]) for v in ops._FROZEN_SHADOWS.values()))

    def _operands(self):
        """The tensors a graph reads: every parameter and buffer of the encoders, the actor (plan proposal) and the
        decoder, and the bf16 shadow of each parameter.  A graph keeps them alive for as long as it exists."""
        keep = []
        for x in self._tensors:
            keep.append(x.detach())
            if isinstance(x, torch.nn.Parameter):
                keep.append(ops.shadow_of(x))
        return keep

    def _capture(self, replan):
        # warm-up on a side stream against copies of the state the step mutates, then restore it
        state = [x for x in (self.plan, self.hidden, self.t, self.plan_value) if x is not None]
        saved = [x.clone() for x in state]
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            self._run(replan)
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        if self._pool is None:
            self._pool = torch.cuda.graph_pool_handle()
        n0 = L.launch_count()
        with torch.cuda.graph(graph, pool=self._pool):
            self._run(replan)
        launches = L.launch_count() - n0
        with torch.no_grad():
            for x, s in zip(state, saved):
                x.copy_(s)
        torch.cuda.synchronize(self.device)
        return graph, launches

    def step(self, obs=None):
        """One control step of every environment.  obs: {modality: (n_envs, 3, H, W)} uint8 frames or normalised
        float32, the same shapes and dtype at every step (None: `static_obs` already holds the observation)."""
        if not self._has_goal.all():
            missing = np.flatnonzero(~self._has_goal).tolist()
            raise ValueError(f"environments {missing} have no goal yet: reset(rows, goal) them before the first step")
        if obs is not None:
            self._check_images(obs, self.obs_mods, self.n, "obs")
            if self.static_obs is None:
                self.static_obs = {k: torch.empty(obs[k].shape, dtype=obs[k].dtype, device=self.device) for k in self.obs_mods}
            for k in self.obs_mods:
                s = self.static_obs[k]
                if obs[k].shape != s.shape or obs[k].dtype != s.dtype:
                    raise ValueError(f"obs[{k!r}] is {tuple(obs[k].shape)} {obs[k].dtype}; this policy's static buffer "
                                     f"is {tuple(s.shape)} {s.dtype}")
                s.copy_(obs[k], non_blocking=True)
        elif self.static_obs is None:
            raise ValueError("no observation: pass obs to the first step")
        replan = bool(self._replan.any())
        self.restart.copy_(torch.from_numpy(self._replan))
        ops.refresh_shadows()          # parameters edited through torch since the last step (checkpoint load, ...)
        if self.use_graphs:
            key = (replan, ops.get_precision())
            sig = self._signature()
            entry = self._graphs.get(key)
            if entry is not None and entry[2] != sig:
                self._graphs.clear()      # every graph reads the same operands: none of them is valid any more
                entry = None
            if entry is None:
                keep = self._operands()          # (creates any frozen shadow before the capture reads it)
                sig = self._signature()
                graph, launches = self._capture(replan)
                # the graph holds raw pointers: keep what it reads alive for as long as the graph exists
                entry = self._graphs[key] = (graph, launches, sig, keep)
                self.captures += 1
            graph, self.launches[key] = entry[:2]
            graph.replay()
        else:
            self._run(replan)
        self._replan[:] = 0
        return self.actions
