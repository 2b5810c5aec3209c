"""Flat-buffer optimiser pieces: one fused clip+Adam kernel launch per parameter group, Polyak over
flat buffers, and the hook where the data-parallel gradient all-reduce plugs in.

Replaces torch.optim.Adam / clip_grad_norm_ / soft_update_from_to at the reference call sites
(play_lmp_for_rl.py:362-368; cql_offline_lightning.py:229-232, 519-542, 553-574)."""
import os

import torch

from . import _lib, ops

_ALIGN = 64   # elements (256 B): keeps every parameter view TMA/float4 friendly


class FlatBuffer:
    """Packs tensors into one contiguous fp32 buffer and re-points their .data at views of it."""

    def __init__(self, tensors, repoint=True):
        self.tensors = list(tensors)
        self.offsets = []
        off = 0
        for t in self.tensors:
            self.offsets.append(off)
            off += (t.numel() + _ALIGN - 1) // _ALIGN * _ALIGN
        self.numel = max(off, _ALIGN)
        dev = self.tensors[0].device if self.tensors else torch.device("cpu")
        self.flat = torch.zeros(self.numel, device=dev, dtype=torch.float32)
        self.views = []
        for t, o in zip(self.tensors, self.offsets):
            v = self.flat[o:o + t.numel()].view(t.shape)
            if repoint:
                v.copy_(t.data)
                t.data = v
            self.views.append(v)


class FlatAdam(torch.optim.Optimizer):
    """Adam over one flat parameter buffer (torch.optim.Adam semantics, no weight decay / amsgrad).

    step(): gather .grad into the flat gradient buffer -> optional `grad_sync(flat_grad)` (the NCCL
    all-reduce of tacorl_b200.parallel) -> optional global-norm clip -> ONE fused Adam kernel.
    `grad_scale` (e.g. 1/world_size) and the clip coefficient are applied inside the kernel."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, max_grad_norm=None):
        params = [p for p in params]
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))
        ps = self.param_groups[0]["params"]
        self.pbuf = FlatBuffer(ps, repoint=True)
        self.flat_grad = torch.zeros_like(self.pbuf.flat)
        self.exp_avg = torch.zeros_like(self.pbuf.flat)
        self.exp_avg_sq = torch.zeros_like(self.pbuf.flat)
        self.grad_views = [self.flat_grad[o:o + p.numel()].view(p.shape) for p, o in zip(ps, self.pbuf.offsets)]
        self.max_grad_norm = max_grad_norm
        self.grad_sync = None       # callable(flat_grad) -> None
        self.grad_scale = 1.0
        self.step_count = 0
        self._sqnorm = torch.zeros(1, device=self.pbuf.flat.device)
        # device-resident step counter: the bias correction stays right when the step is replayed from a CUDA graph
        self._step_dev = (torch.zeros(1, dtype=torch.int32, device=self.pbuf.flat.device)
                          if self.pbuf.flat.is_cuda else None)
        # bf16 twin of the parameters for the tensor-core operands: written by the Adam kernel; ops.shadow_of() re-casts a
        # parameter's slice lazily when a torch-side in-place edit (load_state_dict, broadcast, manual init) moved the
        # parameter's or the flat buffer's version counter
        self.shadow = None
        self._pver = {}
        self._pnumel = {p.data_ptr(): p.numel() for p in ps}
        self._pparam = {p.data_ptr(): p for p in ps}       # slot hand-out checks the owning parameter's .grad
        self._flat_version = self.pbuf.flat._version
        self._slots_taken = set()
        self._ranges = []          # (param lo, param hi, element lo, element hi) runs already exchanged / updated this step
        self._pre = []             # runs whose exchange was started ahead of their update (begin_exchange_only)
        if self.pbuf.flat.is_cuda:
            self.shadow = torch.zeros(self.pbuf.numel, device=self.pbuf.flat.device, dtype=torch.bfloat16)
            ops.register_shadow_owner(self)
            ops.register_grad_owner(self)

    @property
    def flat_params(self):
        return self.pbuf.flat

    def _range_of(self, params):
        ids = {id(p) for p in params}
        idx = [i for i, p in enumerate(self.param_groups[0]["params"]) if id(p) in ids]
        if not idx:
            return None
        lo, hi = min(idx), max(idx)
        assert hi - lo + 1 == len(idx), "overlapped sync needs a contiguous run of parameters"
        ps = self.param_groups[0]["params"]
        end = self.pbuf.offsets[hi + 1] if hi + 1 < len(ps) else self.pbuf.numel
        return lo, hi + 1, self.pbuf.offsets[lo], end

    def begin_exchange_only(self, params):
        """Data parallel only: start the all-reduce of `params` (a contiguous run whose gradients are final) now and leave
        their update to the begin_overlapped_sync() / step() call that covers them later.  Used for a sub-network whose
        backward finishes long before the rest (the action decoder: its exchange then hides under the plan recogniser's
        BPTT, where only the collective's own channel SMs are taken from nobody)."""
        r = self._range_of(params)
        if r is None or self.grad_sync is None or not self.pbuf.flat.is_cuda:
            return
        lo, hi, e0, e1 = r
        if any(not (hi <= a or b <= lo) for a, b, _, _ in self._ranges + self._pre):
            return
        ops.join_pending_grads(self.pbuf.flat.device)    # the exchange reads the slice in the current stream's order
        self.gather_grads(lo, hi)
        if self.sm_reserve:
            _lib.lib().tacorl_set_sm_reserve(int(self.sm_reserve))
            self._reserved = True
        self.grad_sync.start(self.flat_grad[e0:e1])
        self._pre.append((lo, hi, e0, e1))

    def begin_overlapped_sync(self, params):
        """Call when the gradients of `params` (a contiguous run: a whole sub-network) are final while backward is
        still running.  Their slice of the flat gradient is gathered; with data parallelism its all-reduce starts on
        the side stream; and -- when no global-norm clip couples the slices -- the Adam update of the slice follows, so
        that exchange AND update hide under the rest of the backward pass.  May be called several times per step with
        disjoint runs (decoder, plan recogniser, ... as their BPTT finishes); step() handles whatever is left."""
        r = self._range_of(params)
        if r is None:
            return
        early = self.early_step and self.max_grad_norm is None and self.pbuf.flat.is_cuda
        if self.grad_sync is None and not early:
            return
        lo, hi, e0, e1 = r
        if any(not (hi <= a or b <= lo) for a, b, _, _ in self._ranges):
            return                                     # (already handled this step)
        if self.grad_sync is not None:     # the exchange reads the slice in the current stream's order
            ops.join_pending_grads(self.pbuf.flat.device)
        # sub-runs whose exchange was started earlier (begin_exchange_only): gathered and on the wire already
        pre = sorted(q for q in self._pre if lo <= q[0] and q[1] <= hi)
        self._pre = [q for q in self._pre if q not in pre]
        plo = lo
        for a, b, _, _ in pre:
            if a > plo:
                self.gather_grads(plo, a)
            plo = b
        if plo < hi:
            self.gather_grads(plo, hi)
        first = not self._ranges
        self._ranges.append((lo, hi, e0, e1))
        if self.grad_sync is not None and self.sm_reserve and self.pbuf.flat.is_cuda:
            _lib.lib().tacorl_set_sm_reserve(int(self.sm_reserve))      # until step(): kernels under the exchange
            self._reserved = True
        if not early:
            x = e0
            for _, _, a, b in pre:
                if a > x:
                    self.grad_sync.start(self.flat_grad[x:a])
                x = b
            if x < e1:
                self.grad_sync.start(self.flat_grad[x:e1])
            return
        dev = self.pbuf.flat.device
        if self._early_stream is None:
            self._early_stream = torch.cuda.Stream(device=dev)
        stream = self._early_stream
        # the update runs on its own stream (later exchanges must not queue behind it), after the gather ...
        stream.wait_stream(torch.cuda.current_stream(dev))
        ops.wait_pending_grads(stream, dev)            # ... and after weight gradients still running beside the BPTT
        if first:
            self.step_count += 1
        # ... and, with data parallelism, bucket by bucket behind the all-reduce: the update of bucket i overlaps the
        # exchange of bucket i + 1 (the exchange keeps its own SMs -- the NCCL channels -- and the update is HBM-bound)
        step = getattr(self.grad_sync, "bucket", None) if (self.grad_sync is not None and self.pipeline_early) else None
        # pieces in update order: the pre-exchanged sub-runs first (their all-reduce is done or well under way), then the
        # rest bucket by bucket
        pieces, x = [], e0
        for _, _, a, b in pre:
            if a > x:
                pieces.append((x, a, True))
            x = b
        if x < e1:
            pieces.append((x, e1, True))
        todo = [(a, b, False) for _, _, a, b in pre]
        for a, b, _ in pieces:
            cs = list(range(a, b, step)) if step else [a]
            todo += [(c, cs[j + 1] if j + 1 < len(cs) else b, True) for j, c in enumerate(cs)]
        for i, (c0, c1, exchange) in enumerate(todo):
            if self.grad_sync is not None:
                if exchange:
                    self.grad_sync.start(self.flat_grad[c0:c1])
                self.grad_sync.wait_on(stream)
            with torch.cuda.stream(stream):
                # full-size grid: measured on the B200, a background-sized grid (one CTA per SM, tacorl_adam_step_range
                # background = 1) does run under the encoder backward, but the convolution kernels it shares the SMs with
                # slow down by more than the update takes (step 3.39 -> 3.57 ms; profiles/r02)
                self._adam_range(c0, c1, increment=first and i == 0, background=self.early_background)
        self._early = True

    # update slices whose gradient is final early on a side stream (see begin_overlapped_sync).  Off by default: it assumes
    # ONE backward pass per step() (no gradient accumulation); runtime.play_lmp_step_fn, which owns that structure, enables it
    early_step = False
    _pre = ()                 # (replaced by a list in __init__) sub-runs whose exchange started before their update was scheduled
    sm_reserve = 0            # SMs the persistent kernels leave to an overlapped exchange (parallel.attach_data_parallel)
    _reserved = False
    early_background = False
    pipeline_early = os.environ.get("TACORL_PIPELINE_EARLY", "1") != "0"   # bucket-wise exchange -> update pipeline
    _early = False
    _early_stream = None

    def _adam_range(self, e0, e1, increment, sq=None, background=False):
        g = self.param_groups[0]
        ops.adam_step(self.pbuf.flat[e0:e1], self.flat_grad[e0:e1], self.exp_avg[e0:e1], self.exp_avg_sq[e0:e1], g["lr"],
                      self.step_count, g["betas"][0], g["betas"][1], g["eps"], self.grad_scale, sq,
                      float(self.max_grad_norm) if self.max_grad_norm is not None else 0.0, self._step_dev,
                      None if self.shadow is None else self.shadow[e0:e1], increment, background)

    def gather_grads(self, lo=0, hi=None):
        ps = self.param_groups[0]["params"][lo:hi]
        dst, src, missing = [], [], []
        for p, gv in zip(ps, self.grad_views[lo:hi]):
            if p.grad is None:
                if p.data_ptr() not in self._slots_taken:   # (a taken slot already holds this pass's gradient)
                    missing.append(gv)
            elif p.grad.data_ptr() != gv.data_ptr():      # else: the backward kernel wrote the slot itself (ops.grad_slot_of)
                dst.append(gv)
                src.append(p.grad)
        if dst:
            torch._foreach_copy_(dst, src)
        for gv in missing:
            gv.zero_()

    def zero_grad(self, set_to_none=True):
        self._slots_taken.clear()
        if not self._early:
            self._ranges, self._pre = [], []
        return super().zero_grad(set_to_none=set_to_none)

    # ---- checkpointing: torch.optim.Adam's layout ({"state": {i: {step, exp_avg, exp_avg_sq}}, "param_groups": [...]}),
    # so that a Lightning checkpoint written with the reference's Adam resumes here and vice versa
    def invalidate_shadow(self):
        """Call after editing parameters through `p.data` (which does not move the version counters ops.shadow_of
        watches): every bf16 twin slice is re-cast on its next use."""
        self._pver.clear()

    @property
    def steps_done(self):
        """Optimiser steps taken so far.  The device-resident counter is the truth: CUDA-graph replays advance it without
        running this object's Python."""
        return int(self._step_dev.item()) if self._step_dev is not None else self.step_count

    def state_dict(self):
        ps = self.param_groups[0]["params"]
        state = {}
        self.step_count = self.steps_done
        if self.step_count > 0:
            for i, (p, o) in enumerate(zip(ps, self.pbuf.offsets)):
                n = p.numel()
                state[i] = {"step": torch.tensor(float(self.step_count)),
                            "exp_avg": self.exp_avg[o:o + n].view(p.shape).clone(),
                            "exp_avg_sq": self.exp_avg_sq[o:o + n].view(p.shape).clone()}
        groups = [{**{k: v for k, v in g.items() if k != "params"}, "params": list(range(len(ps)))}
                  for g in self.param_groups]
        return {"state": state, "param_groups": groups}

    @torch.no_grad()
    def load_state_dict(self, sd):
        ps = self.param_groups[0]["params"]
        saved = sd["param_groups"][0]
        assert len(saved["params"]) == len(ps), "optimizer state_dict holds a different number of parameters"
        for k in ("lr", "betas", "eps"):
            if k in saved:
                self.param_groups[0][k] = tuple(saved[k]) if k == "betas" else saved[k]
        self.exp_avg.zero_()
        self.exp_avg_sq.zero_()
        steps = set()
        for i, (p, o) in enumerate(zip(ps, self.pbuf.offsets)):
            st = sd["state"].get(i, sd["state"].get(str(i)))
            if st is None:
                continue
            n = p.numel()
            self.exp_avg[o:o + n].copy_(st["exp_avg"].reshape(-1))
            self.exp_avg_sq[o:o + n].copy_(st["exp_avg_sq"].reshape(-1))
            steps.add(int(float(st["step"])))
        assert len(steps) <= 1, f"per-parameter step counts differ ({sorted(steps)}): not one flat Adam group"
        self.step_count = steps.pop() if steps else 0
        if self._step_dev is not None:
            self._step_dev.fill_(self.step_count)
        self.invalidate_shadow()

    def snapshot(self):
        """Everything a step mutates (parameters, moments, step counters): see runtime.GraphedTrainStep."""
        return {"p": self.pbuf.flat.clone(), "m": self.exp_avg.clone(), "v": self.exp_avg_sq.clone(),
                "step": self.steps_done, "shadow": None if self.shadow is None else self.shadow.clone()}

    @torch.no_grad()
    def restore(self, snap):
        self.pbuf.flat.copy_(snap["p"])
        self.exp_avg.copy_(snap["m"])
        self.exp_avg_sq.copy_(snap["v"])
        self.step_count = snap["step"]
        if self._step_dev is not None:
            self._step_dev.fill_(self.step_count)
        if self.shadow is not None:
            self.shadow.copy_(snap["shadow"])

    @torch.no_grad()
    def step(self, closure=None, gathered=False):
        loss = closure() if closure is not None else None
        if self.pbuf.flat.is_cuda:
            ops.join_pending_grads(self.pbuf.flat.device)
        self._slots_taken.clear()
        if self._reserved:                         # the kernels that ran under the overlapped exchange are all launched
            _lib.lib().tacorl_set_sm_reserve(0)
            self._reserved = False
        n, numel = len(self.param_groups[0]["params"]), self.pbuf.numel
        done = sorted(self._ranges)
        left_pre = sorted(self._pre)               # exchanged ahead of time, never covered by an early update
        self._ranges, self._pre = [], []
        # complement of the runs handled early, in parameter-index space and in element space
        rest_p, rest_e, p0, x0 = [], [], 0, 0
        for lo, hi, e0, e1 in sorted(done + left_pre):
            if lo > p0:
                rest_p.append((p0, lo))
            if e0 > x0:
                rest_e.append((x0, e0))
            p0, x0 = hi, e1
        if p0 < n:
            rest_p.append((p0, n))
        if x0 < numel:
            rest_e.append((x0, numel))
        if not gathered:
            for a, b in rest_p:
                self.gather_grads(a, b)
        if self.grad_sync is not None:
            for a, b in rest_e:
                self.grad_sync.start(self.flat_grad[a:b])
            self.grad_sync.finish()
        if self._early:                            # some slices were updated early: only the remaining ones are left
            for a, b in rest_e + [(e0, e1) for _, _, e0, e1 in left_pre]:
                self._adam_range(a, b, increment=False)
            torch.cuda.current_stream(self.pbuf.flat.device).wait_stream(self._early_stream)
            self._early = False
            return loss
        assert not (done or left_pre) or self.grad_sync is not None
        self.step_count += 1
        sq = None
        if self.max_grad_norm is not None:
            sq = ops.sqnorm(self.flat_grad, self._sqnorm)
        self._adam_range(0, numel, increment=True, sq=sq)
        return loss

    def set_grad(self, flat_values):
        """Directly provide the flat gradient (single-element groups such as log_alpha)."""
        self.flat_grad[:flat_values.numel()].copy_(flat_values.reshape(-1))


def polyak_update(target_buf: FlatBuffer, source_flat: torch.Tensor, tau: float):
    """target <- (1 - tau) target + tau source over two flat buffers with the SAME layout (every source parameter
    trainable, cql_offline_lightning.py:229-232 pairs .parameters() by position)."""
    assert target_buf.flat.numel() == source_flat.numel(), (
        f"Polyak: target buffer ({target_buf.flat.numel()}) and source buffer ({source_flat.numel()}) differ: a frozen "
        "q-network parameter changes the flat layout")
    ops.polyak_update(target_buf.flat, source_flat, tau)
