"""Mirror of PlayLMP, /root/reference/src/tacorl/modules/play_lmp/play_lmp_for_rl.py:17-368.
Same ctor kwargs (config/module/play_lmp_for_rl.yaml), same training_step contract (returns the
scalar total loss; logs the same metric names), same state_dict layout (SURVEY.md Appendix B)."""
from typing import Dict, List, Optional

import os

import torch

from ... import ops
from ...optim import FlatAdam
from ...utils import rng
from ...utils.config import instantiate, to_container
from ...utils.distributions import TanhNormal
from ...utils.lightning import LightningModule


class PlayLMP(LightningModule):
    def __init__(self, env: dict = {}, actor: dict = {}, plan_proposal: dict = {}, plan_recognition: dict = {},
                 perceptual_encoder: dict = {}, goal_encoder: dict = {}, action_decoder: dict = {},
                 transform_manager: dict = {}, dataloader: dict = {}, kl_beta: float = 1e-3,
                 kl_balancing: bool = True, add_random_plan_loss: bool = False, kl_alpha: float = 0.8,
                 lr: float = 1e-4, plan_proposal_obs_modalities: List[str] = [],
                 plan_proposal_goal_modalities: List[str] = [], plan_recognition_modalities: List[str] = [],
                 action_decoder_modalities: List[str] = [], real_world: bool = False, *args, **kwargs):
        super().__init__(*args, **kwargs)
        # The simulator (env / make_env, :46-49) is outside the training hot path; rollout callbacks
        # that need it attach their own env.
        self.real_world = real_world
        self.env_cfg = env
        self.env = None
        self.add_random_plan_loss = add_random_plan_loss
        self.plan_proposal_obs_modalities = list(plan_proposal_obs_modalities)
        self.plan_proposal_goal_modalities = list(plan_proposal_goal_modalities)
        self.plan_recognition_modalities = list(plan_recognition_modalities)
        self.action_decoder_modalities = list(action_decoder_modalities)
        all_modalities = (self.plan_proposal_obs_modalities + self.plan_proposal_goal_modalities
                          + self.plan_recognition_modalities + self.action_decoder_modalities)
        self.all_modalities = sorted(set(all_modalities), key=all_modalities.index)
        self.transform_manager = instantiate(transform_manager) if transform_manager else None
        self.actor_cfg = actor
        self.plan_proposal_cfg = plan_proposal
        self.plan_recognition_cfg = plan_recognition
        self.perceptual_encoder_cfg = perceptual_encoder
        self.goal_encoder_cfg = goal_encoder
        self.action_decoder_cfg = action_decoder
        self.build_networks()
        self.lr = lr
        self.dataloader = dataloader
        self.kl_beta = kl_beta
        self.completed_tasks_by_idx = {}
        self.kl_balancing = kl_balancing
        self.kl_alpha = kl_alpha
        self.save_hyperparameters()

    def build_networks(self):                                                     # :80-130
        pe_cfg = to_container(self.perceptual_encoder_cfg)
        pe_cfg["modalities"] = self.all_modalities
        self.perceptual_encoder = instantiate(pe_cfg)
        pp_state_dim = self.perceptual_encoder.calc_state_dim(modalities=self.plan_proposal_obs_modalities)
        pp_goal_dim = self.perceptual_encoder.calc_state_dim(modalities=self.plan_proposal_goal_modalities)
        pr_dim = self.perceptual_encoder.calc_state_dim(modalities=self.plan_recognition_modalities)
        ge_cfg = to_container(self.goal_encoder_cfg)
        ge_cfg["in_features"] = pp_goal_dim
        ge_cfg["out_features"] = pp_goal_dim
        self.goal_encoder = instantiate(ge_cfg)
        pr_cfg = to_container(self.plan_recognition_cfg)
        pr_cfg["state_dim"] = pr_dim
        self.plan_recognition = instantiate(pr_cfg)
        pp_cfg = to_container(self.plan_proposal_cfg)
        pp_cfg["state_dim"] = pp_state_dim
        pp_cfg["goal_dim"] = ge_cfg["out_features"]
        if "Actor" in pp_cfg["_target_"].split(".")[-1]:
            pp_cfg["action_dim"] = self.plan_recognition.latent_plan_dim
        self.plan_proposal = instantiate(pp_cfg)
        ad_cfg = to_container(self.action_decoder_cfg)
        ad_cfg["state_dim"] = self.perceptual_encoder.calc_state_dim(modalities=self.action_decoder_modalities)
        ad_cfg["goal_dim"] = ge_cfg["out_features"]
        self.action_decoder = instantiate(ad_cfg)

    def compute_action_loss(self, emb_states, actions, latent_plan, stage: str = "train",
                            log_name_prefix: str = "", latent_goal: Optional[torch.Tensor] = None):  # :132-185
        action_loss, pred_actions = self.action_decoder.loss_and_act(
            latent_plan=latent_plan, perceptual_emb=emb_states[:, :-1], actions=actions[:, :-1])
        self.log(f"{stage}/{log_name_prefix}action_loss", action_loss, on_step=True, on_epoch=True, sync_dist=True)
        # gripper accuracy (:165-176) is produced by the sampling kernel
        self.log(f"{stage}/{log_name_prefix}gripper_accuracy", self.action_decoder.last_gripper_accuracy,
                 on_step=True, on_epoch=True, sync_dist=True)
        return action_loss

    def get_emb_states(self, states, modalities: List[str] = []):                 # :187-198 (no in-place rebind)
        bs, seq_len = list(states.values())[0].shape[:2]
        flat = {k: v.reshape(bs * seq_len, *v.shape[2:]) for k, v in states.items()}
        emb = self.perceptual_encoder.get_state_from_observation(observation=flat, modalities=modalities,
                                                                 cat_output=False)
        return {k: v.view(bs, seq_len, -1) for k, v in emb.items()}

    @staticmethod
    def _cat(tensors):
        return tensors[0] if len(tensors) == 1 else torch.cat(tensors, dim=-1)

    def process_batch(self, batch):                                               # :200-219
        emb_states = self.get_emb_states(batch["states"], modalities=self.all_modalities)
        self._overlap_grad_sync(emb_states)
        pp_state = self._cat([emb_states[k][:, 0] for k in self.plan_proposal_obs_modalities])
        pp_goal = self._cat([emb_states[k][:, -1] for k in self.plan_proposal_goal_modalities])
        pr_states = self._cat([emb_states[k] for k in self.plan_recognition_modalities])
        if self.early_subnet_sync and self._sync_active():
            pr_states = pr_states.view_as(pr_states)      # own autograd node: its gradient = "the recogniser's BPTT is done"
            self._sync_when_grad_of(pr_states, [self.plan_recognition])
        pr_dist = self.plan_recognition(pr_states)

        # Goal encoder and plan proposal on a forked stream, so that autograd runs their backward there too: it then waits
        # only on the KL gradient and runs beside the decoder's BPTT instead of after the recogniser's.  Forked after the
        # recogniser, whose two-lane layer-0 recurrence leaves no room for the chains' 32 CTAs.
        def proposal():
            goal = self.goal_encoder(pp_goal)
            return goal, self.plan_proposal.get_dist(pp_state, goal)
        pp_goal, pp_dist = ops.forked(proposal, pp_state.device) if torch.is_grad_enabled() else proposal()
        return emb_states, pp_dist, pr_dist, pp_goal

    def compute_loss(self, batch, stage: str = "train"):                          # :221-257
        emb_states, pp_dist, pr_dist, lat_goal = self.process_batch(batch)
        ad_states = self._cat([emb_states[k] for k in self.action_decoder_modalities])
        latent_plan = pr_dist.rsample()
        self._sync_when_grad_of(latent_plan, [self.action_decoder])       # decoder BPTT done -> its slice can go
        self._exchange_when_grad_of(latent_plan, [self.action_decoder])
        mean_shape = pr_dist.normal.mean.shape if isinstance(pr_dist, TanhNormal) else pr_dist.mean.shape
        dec = self.action_decoder
        if self.add_random_plan_loss or not hasattr(dec, "loss_and_act_two_plans"):
            action_loss = self.compute_action_loss(emb_states=ad_states, actions=batch["actions"],
                                                   latent_plan=latent_plan, stage=stage, latent_goal=lat_goal)
            random_plan = rng.uniform(mean_shape, -1.0, 1.0, lat_goal.device)
            rng.uniform(lat_goal.shape, -1.0, 1.0, lat_goal.device)   # the reference also draws an (unused) goal
            rp_loss = self.compute_action_loss(ad_states, batch["actions"], random_plan, stage, "random_plan_")
        else:
            # sampled plan and random plan (logging only, :243-256) share ONE batched decoder pass; the noise is
            # drawn in the reference's order: _sample(u1,u2) -> random plan -> (unused) random goal -> _sample
            Bn, Tn = ad_states.shape[0], ad_states.shape[1] - 1
            noise = dec._draw_sample_noise(Bn, Tn, lat_goal.device)
            random_plan = rng.uniform(mean_shape, -1.0, 1.0, lat_goal.device)
            rng.uniform(lat_goal.shape, -1.0, 1.0, lat_goal.device)
            noise_rp = dec._draw_sample_noise(Bn, Tn, lat_goal.device)
            (action_loss, _, acc), (rp_loss, _, acc_rp) = dec.loss_and_act_two_plans(
                latent_plan, random_plan, ad_states[:, :-1], batch["actions"][:, :-1], noise, noise_rp)
            for prefix, l_, a_ in (("", action_loss, acc), ("random_plan_", rp_loss, acc_rp)):
                self.log(f"{stage}/{prefix}action_loss", l_, on_step=True, on_epoch=True, sync_dist=True)
                self.log(f"{stage}/{prefix}gripper_accuracy", a_, on_step=True, on_epoch=True, sync_dist=True)
        # after the decoder: autograd orders a pass's backward by creation, latest first, so the KL gradient (all the plan
        # proposal's backward waits on) is issued before the decoder's BPTT
        kl_loss = self.compute_kl_loss(pr_dist=pr_dist, pp_dist=pp_dist, stage=stage)
        total_loss = kl_loss + action_loss
        if self.add_random_plan_loss:
            total_loss = total_loss - rp_loss
        return total_loss, pp_dist

    def compute_kl_loss(self, pr_dist, pp_dist, stage: str = "train"):            # :259-301
        prior = pp_dist.normal if isinstance(pp_dist, TanhNormal) else pp_dist
        posterior = pr_dist.normal if isinstance(pr_dist, TanhNormal) else pr_dist
        kl_loss = ops.kl_balanced(posterior.mean, posterior.stddev, prior.mean, prior.stddev, self.kl_alpha,
                                  self.kl_balancing)
        kl_loss_scaled = kl_loss * self.kl_beta
        self.log(f"{stage}/kl_loss", kl_loss, on_step=True, on_epoch=True, sync_dist=True)
        self.log(f"{stage}/kl_loss_scaled", kl_loss_scaled, on_step=True, on_epoch=True, sync_dist=True)
        return kl_loss_scaled

    def set_kl_beta(self, kl_beta):
        self.kl_beta = kl_beta

    def training_step(self, batch: Dict[str, torch.Tensor], batch_idx=0):         # :307-317
        total_loss, _ = self.compute_loss(batch, stage="train")
        self.log("train/total_loss", total_loss, on_step=True, on_epoch=True, sync_dist=True)
        return total_loss

    def validation_step(self, batch, batch_idx=0):                                # :319-348
        with torch.no_grad():
            total_loss, pp_dist = self.compute_loss(batch, stage="validation")
        self.log("validation/total_loss", total_loss, on_step=True, on_epoch=True, sync_dist=True)
        return {"idx": batch.get("idx"), "sampled_plan_pp": pp_dist.sample()}

    def configure_optimizers(self):                                               # :362-368
        self._flat_opt = FlatAdam(filter(lambda p: p.requires_grad, self.parameters()), lr=self.lr)
        return self._flat_opt

    _flat_opt = None

    def _sync_active(self):
        opt = self._flat_opt
        return opt is not None and torch.is_grad_enabled() and (opt.grad_sync is not None or opt.early_step)

    # Exchange / update the decoder's and the recogniser's slices as soon as their own BPTT finishes (instead of when
    # the embeddings' gradient exists).  Off: measured at N = 2, the extra NCCL / Adam grids then run while the persistent
    # recurrence kernels of the other sub-network need 120-128 co-resident SMs, and the step gets slower (3.51 -> 3.67 ms).
    early_subnet_sync = False

    def _sync_when_grad_of(self, tensor, modules):
        """Start the gradient exchange / early update of `modules`' parameters as soon as the gradient w.r.t. `tensor`
        (their only input that requires one) exists, i.e. their backward pass is complete."""
        if not self.early_subnet_sync or not self._sync_active() or not tensor.requires_grad:
            return
        opt = self._flat_opt
        ids = set()
        for m in modules:
            ids |= {id(p) for p in m.parameters()}
        params = [p for p in opt.param_groups[0]["params"] if id(p) in ids]

        def hook(grad):
            opt.begin_overlapped_sync(params)
            return None

        tensor.register_hook(hook)

    # Data parallel: put the action decoder's gradients (13 M of 47 M parameters) on the wire as soon as its BPTT is done;
    # the exchange then runs under the plan recogniser's BPTT (its 16 channel CTAs fit beside the recurrence's 128) and
    # only two of three buckets are left when the embeddings' gradient exists.  Update still at the embeddings' hook.
    # Opt-in: measured at N = 2 (profiles/r02/timeline_n2_dec1.json) the early exchange does hide (187 us under the BPTT),
    # but the remaining buckets still queue behind the early Adam grids for their SMs and the step does not get shorter
    # (3.47 vs 3.42 ms).
    early_decoder_exchange = os.environ.get("TACORL_EARLY_DECODER_EXCHANGE", "0") == "1"

    def _exchange_when_grad_of(self, tensor, modules):
        opt = self._flat_opt
        if (not self.early_decoder_exchange or opt is None or opt.grad_sync is None or not torch.is_grad_enabled()
                or not tensor.requires_grad or not getattr(opt, "sm_reserve", 0) or opt.sm_reserve + 128 > 148):
            return
        ids = set()
        for m in modules:
            ids |= {id(p) for p in m.parameters()}
        params = [p for p in opt.param_groups[0]["params"] if id(p) in ids]

        def hook(grad):
            opt.begin_exchange_only(params)
            return None

        tensor.register_hook(hook)

    def _overlap_grad_sync(self, emb_states):
        """Everything behind the vision encoders (RNNs, decoder, MLPs = 99.7 % of the parameters) has its final
        gradient before the encoders' backward starts.  A hook on the embeddings starts the all-reduce of that slice
        (data parallel) and its Adam update (optimizer.early_step) at exactly that moment, on side streams, so both
        overlap the encoder backward.  (The decoder and the plan recogniser are started even earlier, as their own
        BPTT finishes: compute_loss / process_batch.)"""
        if not self._sync_active():
            return
        opt = self._flat_opt
        enc_ids = {id(p) for p in self.perceptual_encoder.parameters()}
        groups, run = [], []
        for p in opt.param_groups[0]["params"]:        # contiguous runs of non-encoder parameters
            if id(p) in enc_ids:
                if run:
                    groups.append(run)
                run = []
            else:
                run.append(p)
        if run:
            groups.append(run)
        pending = [len(emb_states)]

        def hook(grad):
            pending[0] -= 1
            if pending[0] == 0:
                for g in groups:
                    # (runs the decoder / recogniser hooks already handled are skipped inside; what is left of a run
                    # that contains them is picked up by step())
                    opt.begin_overlapped_sync(g)
            return None

        for v in emb_states.values():
            if v.requires_grad:
                v.register_hook(hook)
            else:
                pending[0] -= 1
