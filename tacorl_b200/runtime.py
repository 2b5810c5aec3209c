"""CUDA-graph execution of a whole training step (forward + backward + all-reduce + optimiser).

The step issues several hundred small launches (per-timestep recurrent GEMMs, per-chunk conv GEMMs, loss
kernels); replaying them from one captured graph removes the host launch / ctypes / autograd overhead that would
otherwise dominate a ~ms step (SURVEY.md §7 "Host overhead").  Noise keeps advancing between replays (the torch
CUDA generator is graph-aware) and the Adam bias correction reads a device-resident step counter."""
import ctypes

import torch


def _clone_to_static(batch, device):
    out = {}
    for k, v in batch.items():
        if isinstance(v, dict):
            out[k] = _clone_to_static(v, device)
        elif torch.is_tensor(v):
            out[k] = v.to(device, non_blocking=True).clone()
        else:
            out[k] = v
    return out


def _tensors(batch):
    for v in batch.values():
        if isinstance(v, dict):
            yield from _tensors(v)
        elif torch.is_tensor(v):
            yield v


def _copy_into(static, batch):
    for k, v in batch.items():
        if isinstance(v, dict):
            _copy_into(static[k], v)
        elif torch.is_tensor(v):
            static[k].copy_(v, non_blocking=True)


def _snapshot(objs):
    return [(o, o.snapshot() if hasattr(o, "snapshot") else o.clone()) for o in objs]


@torch.no_grad()
def _restore(snaps):
    for o, s in snaps:
        if hasattr(o, "restore"):
            o.restore(s)
        else:
            o.copy_(s)


class GraphedTrainStep:
    """step_fn(static_batch) must run one full optimisation step and return a scalar device tensor (or None).
    Usage:  g = GraphedTrainStep(step_fn, example_batch); loss = g(next_batch)

    A captured graph freezes everything the HOST decided while it was recorded: Python branches (TACO-RL's
    `current_epoch < bc_epochs` actor loss, `finetune_action_decoder`) and scalars passed by value (`kl_beta`, learning
    rates).  `mode_key` (default: `step_fn.mode_key`) returns a hashable summary of that host state; one graph is kept
    per distinct key and a new one is captured the first time a key is seen, so crossing `bc_epochs` or calling
    `set_kl_beta` takes effect on the next call.  `preserve` (default: `step_fn.preserve`) lists the optimisers /
    tensors a step mutates: they are saved before the warm-up steps a capture needs and restored afterwards, so
    building a graph does not train on the example batch."""

    def __init__(self, step_fn, example_batch, device=None, warmup=3, mode_key=None, preserve=None, buffers=1,
                 source=None):
        """buffers=2: two sets of static input buffers, one captured graph per set (sharing one memory pool), used
        alternately: `prefetch()` copies the next batch host->device straight into the set the running step is NOT
        reading, so a host-fed loop needs no staging->static device copy between replays.
        source: a tacorl_b200.replay.DeviceReplay.  Every capture records `source.sample()` ahead of the step, so a
        replay draws, assembles and trains with no host work and no host->device copy; `example_batch` may be None and
        calls take no batch.  The source's step counter joins `preserve`: the warm-up steps consume no draws."""
        device = device or torch.device("cuda", torch.cuda.current_device())
        self.device = device
        self.source = source
        if source is not None:
            if int(buffers) != 1:
                raise ValueError("a replay source fills its own buffers: buffers must be 1")
            self.statics = [source.batch()]
            inner = step_fn

            def step_fn(static, _inner=inner):
                source.sample()
                return _inner(static)
            for attr in ("mode_key", "preserve"):
                if hasattr(inner, attr):
                    setattr(step_fn, attr, getattr(inner, attr))
        else:
            self.statics = [_clone_to_static(example_batch, device) for _ in range(max(1, int(buffers)))]
        self._cur = 0
        self.step_fn = step_fn
        self.warmup = warmup
        self.mode_key = mode_key if mode_key is not None else getattr(step_fn, "mode_key", None)
        self.preserve = preserve if preserve is not None else getattr(step_fn, "preserve", None)
        if source is not None:
            inner_preserve = self.preserve
            self.preserve = lambda: (list(inner_preserve()) if inner_preserve is not None else []) + source.preserve()
        self._graphs = {}
        self._pool = None
        self.replays = 0
        self.captures = 0
        self._select(self._key())

    @property
    def static(self):
        return self.statics[self._cur]

    def _key(self):
        return self.mode_key() if self.mode_key is not None else None

    def _capture(self, static):
        from . import _lib
        device = self.device
        snaps = _snapshot(self.preserve()) if self.preserve is not None else None
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            for _ in range(self.warmup):
                self.step_fn(static)
        torch.cuda.current_stream(device).wait_stream(side)
        torch.cuda.synchronize(device)
        graph = torch.cuda.CUDAGraph()
        if self._pool is None:
            self._pool = torch.cuda.graph_pool_handle()      # graphs of one runner never run concurrently: one pool
        n0 = _lib.launch_count()
        with torch.cuda.graph(graph, pool=self._pool):
            out = self.step_fn(static)
            out = out.detach() if torch.is_tensor(out) else None
        # kernels of libtacorl_b200.so recorded in the graph = launched again by every replay
        launches = _lib.launch_count() - n0
        if snaps is not None:
            _restore(snaps)
            torch.cuda.synchronize(device)
        self.captures += 1
        return graph, out, launches

    def _select(self, key):
        k = (key, self._cur)
        if k not in self._graphs:
            self._graphs[k] = self._capture(self.statics[self._cur])
        self.graph, self.out, self.launches_per_replay = self._graphs[k]
        self._active_key = k

    def __call__(self, batch=None):
        """Returns the step's output tensor; with buffers > 1 it is only valid until the next call (shared pool)."""
        main = torch.cuda.current_stream()
        if batch is not None and self.source is not None:
            raise ValueError("this step samples its batch from its replay source: call it without a batch")
        if batch is not None:
            _copy_into(self.static, batch)
        elif self._staged:
            main.wait_event(self._ready)              # the H2D of this step's inputs
            if len(self.statics) > 1:
                self._cur = self._staged_buf           # ... which went straight into the other buffer set
            else:
                _copy_into(self.static, self._staging)
                self._consumed.record(main)
            self._staged = False
        key = self._key()
        if (key, self._cur) != self._active_key:
            self._select(key)
        from . import ops
        ops.refresh_shadows()      # parameters edited through torch since the last replay (checkpoint load, ...)
        self.graph.replay()
        if len(self.statics) > 1 and self._free is not None:
            self._free[self._cur].record(main)         # this buffer set may be refilled once the replay has finished
        self.replays += 1
        return self.out

    _staged = False
    _staging = None
    _free = None

    def prefetch(self, host_batch):
        """Start the host->device copy of the NEXT step's (pinned) batch on a side stream so it overlaps the
        step that is running; the following `__call__()` consumes it (double buffering, like a pinned
        DataLoader with non_blocking copies)."""
        if self._staging is None:
            self._copy_stream = torch.cuda.Stream()
            self._ready = torch.cuda.Event()
            if len(self.statics) > 1:
                self._staging = True
                self._free = [torch.cuda.Event() for _ in self.statics]
                for e in self._free:
                    e.record(torch.cuda.current_stream())
            else:
                self._staging = _clone_to_static(self.static, next(iter(_tensors(self.static))).device)
                self._consumed = torch.cuda.Event()
                self._consumed.record(torch.cuda.current_stream())
        with torch.cuda.stream(self._copy_stream):
            if len(self.statics) > 1:
                target = (self._cur + 1) % len(self.statics)
                self._copy_stream.wait_event(self._free[target])
                _copy_into(self.statics[target], host_batch)
                self._staged_buf = target
            else:
                self._copy_stream.wait_event(self._consumed)
                _copy_into(self._staging, host_batch)
            self._ready.record(self._copy_stream)
        self._staged = True


def play_lmp_step_fn(module, optimizer, early_step=True):
    """One PlayLMP optimiser step.  early_step: this function runs exactly one backward pass per step(), so the update
    of the parameters behind the encoders may start as soon as their gradients are final (FlatAdam.early_step)."""
    optimizer.early_step = bool(early_step)
    import os
    if os.environ.get("TACORL_EARLY_SUBNET") is not None:      # experiment switches (scripts/early_adam_sweep.sh)
        module.early_subnet_sync = os.environ["TACORL_EARLY_SUBNET"] == "1"
    if os.environ.get("TACORL_EARLY_BG") is not None:
        optimizer.early_background = os.environ["TACORL_EARLY_BG"] == "1"

    def step(batch):
        optimizer.zero_grad(set_to_none=True)
        loss = module.training_step(batch, 0)
        loss.backward()
        optimizer.step()
        return loss
    step.mode_key = lambda: (float(module.kl_beta), float(optimizer.param_groups[0]["lr"]), bool(module.training))
    step.preserve = lambda: [optimizer]
    return step


def tacorl_step_fn(module):
    """Step function of a manual-optimisation module: TACORL or the flat CQL_Offline baseline."""
    def step(batch):
        module.training_step(batch)
        return module.logged.get("train/q1_loss")
    opts = module.optimizers()
    step.mode_key = lambda: (module.current_epoch < module.bc_epochs, bool(getattr(module, "finetune_action_decoder", False)),
                             tuple(float(o.param_groups[0]["lr"]) for o in opts), bool(module.training))
    step.preserve = lambda: list(opts) + [b.flat for b in (module._target_bufs or ())]
    return step


def item_weighted_means(keys, totals):
    """Epoch value of every logged validation scalar: `totals` holds one (sums, count) vector per rank, sums[i] =
    sum over the rank's batches of n_b * mean_b of keys[i], count = sum of n_b.  Ranks are added before dividing, as
    Lightning aggregates `self.log(..., on_epoch=True, sync_dist=True)`.  Pure host function."""
    rows = [[float(x) for x in t] for t in totals]
    if not rows or any(len(r) != len(keys) + 1 for r in rows):
        raise ValueError(f"expected (sums, count) vectors of {len(keys) + 1} entries")
    total = [sum(col) for col in zip(*rows)]
    count = total[-1]
    if count <= 0:
        raise ValueError("no validation item was evaluated")
    return {k: total[i] / count for i, k in enumerate(keys)}


class MetricsAccumulator:
    """Device fp64 (sums, count) of the `prefix` scalars a module logs: `add(logged, n)` is one launch
    (tacorl_metrics_accumulate, graph-capturable, no host copy) that adds n * value to each sum and n to the count.
    The keys are fixed by the first add().  `read()` is the only device-to-host copy."""

    def __init__(self, device, prefix="validation/"):
        from . import _lib
        device = torch.device(device)
        self.device = device if device.index is not None else torch.device("cuda", torch.cuda.current_device())
        self.prefix = prefix
        self.keys = None
        self.acc = torch.zeros(_lib.METRICS_MAX + 1, dtype=torch.float64, device=self.device)

    def reset(self):
        self.acc.zero_()

    def add(self, logged, n):
        from . import _lib
        if self.keys is None:
            self.keys = sorted(k for k in logged if k.startswith(self.prefix))
            if not self.keys:
                raise ValueError(f"the step logged no '{self.prefix}*' scalar")
            if len(self.keys) > _lib.METRICS_MAX:
                raise ValueError(f"{len(self.keys)} metrics; at most {_lib.METRICS_MAX} are accumulated")
        m = _lib.Metrics()
        for i, k in enumerate(self.keys):
            v = logged.get(k)
            if not torch.is_tensor(v) or v.numel() != 1 or v.device != self.device:
                raise ValueError(f"{k}: expected a one-element tensor on {self.device}, got {v!r}")
            if v.dtype != torch.float32:
                v = v.float()
                logged[k] = v                         # keeps the converted value alive while the launch reads it
            m.value[i] = v.data_ptr()
        m.k, m.n = len(self.keys), int(n)
        _lib.call("tacorl_metrics_accumulate", ctypes.byref(m), _lib.ptr_any(self.acc), _lib.stream())

    def totals(self):
        """The (sums, count) vector on the device."""
        return self.acc[:len(self.keys or ()) + 1]

    def read(self, totals=None):
        """{key: item-weighted mean} from the device vector (one device-to-host copy)."""
        if self.keys is None:
            raise ValueError("no validation batch was evaluated")
        t = (self.totals() if totals is None else totals).cpu().tolist()
        return item_weighted_means(self.keys, [t])


def validation_step_fn(module, accumulator):
    """One validation batch: `module.validation_step(batch)` under no_grad, then the accumulate launch with the batch's
    item count (its rows).  Same contract as play_lmp_step_fn / tacorl_step_fn, so GraphedTrainStep replays it."""
    def step(batch):
        with torch.no_grad():
            module.validation_step(batch, 0)
        accumulator.add(module.logged, batch["actions"].shape[0])
    # host state the validation forward reads: TACO-RL's BC actor loss below bc_epochs, PlayLMP's kl_beta by value
    step.mode_key = lambda: (module.current_epoch < getattr(module, "bc_epochs", 0), float(getattr(module, "kl_beta", 0.0)),
                             bool(getattr(module, "finetune_action_decoder", False)), bool(module.training))
    step.preserve = lambda: [accumulator.acc]
    return step
