"""CUDA-graph execution of a whole training step (forward + backward + all-reduce + optimiser).

The step issues several hundred small launches (per-timestep recurrent GEMMs, per-chunk conv GEMMs, loss
kernels); replaying them from one captured graph removes the host launch / ctypes / autograd overhead that would
otherwise dominate a ~ms step (SURVEY.md §7 "Host overhead").  Noise keeps advancing between replays (the torch
CUDA generator is graph-aware) and the Adam bias correction reads a device-resident step counter."""
import csv
import ctypes
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist


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


def assign_columns(keys, names):
    """Appends to `keys` (in place) every name it lacks, in order: a key keeps its column for good, because captured
    graphs hold the ring's pointers.  Refuses more than METRICS_MAX keys.  Pure host function."""
    from . import _lib
    for k in names:
        if k not in keys:
            if len(keys) == _lib.METRICS_MAX:
                raise ValueError(f"the step logs more than {_lib.METRICS_MAX} 'train/*' scalars ({k!r} is one too "
                                 f"many); at most {_lib.METRICS_MAX} are recorded")
            keys.append(k)
    return keys


def epoch_means(keys, totals):
    """Epoch mean of every recorded training scalar.  `totals` holds one vector per rank: METRICS_MAX fp64 sums, then
    METRICS_MAX counts (sums[i]: the values of keys[i] over the steps that logged it; counts[i]: those steps).  Ranks
    are added before dividing, as Lightning aggregates `self.log(..., on_epoch=True, sync_dist=True)`; a key no step of
    the epoch logged has no mean.  Pure host function."""
    from . import _lib
    M = _lib.METRICS_MAX
    rows = [[float(x) for x in t] for t in totals]
    if not rows or any(len(r) != 2 * M for r in rows):
        raise ValueError(f"expected (sums, counts) vectors of {2 * M} entries")
    total = [sum(col) for col in zip(*rows)]
    return {k: total[i] / total[M + i] for i, k in enumerate(keys) if total[M + i] > 0}


class RingBook:
    """Host side of the metrics ring: the device counter puts the n-th recorded step (n counts from 0 since the ring
    was made) in row n % (2 * half).  `advance` notes each step's (global step, epoch) and hands over a range when its
    step fills a half; `take` hands over whatever is not handed over yet (epoch and fit end).  A range never spans two
    halves, since a half boundary always ends one.  Pure host class."""

    def __init__(self, half):
        self.half, self.rows = int(half), 2 * int(half)
        self.n = 0               # steps recorded
        self.taken = 0           # steps handed over for read-back
        self._steps, self._epochs = [], []

    def advance(self, global_step, epoch):
        """One more recorded step; returns `take()` when it filled a half, else None."""
        self._steps.append(int(global_step))
        self._epochs.append(int(epoch))
        self.n += 1
        return self.take() if self.n % self.half == 0 else None

    def take(self):
        """(first ring row, global steps, epochs) of steps [taken, n), or None when there are none."""
        if self.taken == self.n:
            return None
        row0 = self.taken % self.rows
        out = (row0, np.asarray(self._steps, np.int64), np.asarray(self._epochs, np.int32))
        self._steps, self._epochs = [], []
        self.taken = self.n
        return out


class TrainHistory:
    """One row per training step, as numpy blocks in the order they were read back: `steps` (global step), `epochs`
    and `values` (len(steps) x len(keys) fp32, NaN where the step did not log the key).  Pure host class."""

    def __init__(self):
        self.keys = []
        self._blocks = []        # (steps, epochs, column index of each value column, values)

    def append(self, keys, steps, epochs, values):
        assign_columns(self.keys, keys)
        cols = np.asarray([self.keys.index(k) for k in keys], np.int64)
        self._blocks.append((np.asarray(steps, np.int64), np.asarray(epochs, np.int32), cols,
                             np.asarray(values, np.float32)[:, :len(keys)]))

    def __len__(self):
        return sum(len(b[0]) for b in self._blocks)

    @property
    def steps(self):
        return np.concatenate([b[0] for b in self._blocks]) if self._blocks else np.zeros(0, np.int64)

    @property
    def epochs(self):
        return np.concatenate([b[1] for b in self._blocks]) if self._blocks else np.zeros(0, np.int32)

    @property
    def values(self):
        out = np.full((len(self), len(self.keys)), np.nan, np.float32)
        r = 0
        for steps, _, cols, vals in self._blocks:
            out[r:r + len(steps), cols] = vals
            r += len(steps)
        return out

    def column(self, key):
        return self.values[:, self.keys.index(key)]


class MetricsCSV:
    """`metrics.csv` in Lightning CSVLogger's layout: a header, then one row per logged step.  Columns: `step`,
    `epoch`, every key (the step's values) and `<key>_epoch` for every key (the epoch means, in one row per epoch at the
    epoch's last step).  Rows of steps >= `start_step` left by an earlier run are dropped (the run resumes from a
    checkpoint written before them) and new rows are appended; a key that is new to the file rewrites it with the
    wider header.  Pure host class."""

    def __init__(self, path, start_step=0):
        self.path = Path(path)
        self.keys, rows = [], []
        if self.path.is_file():
            with open(self.path, newline="") as f:
                r = csv.DictReader(f)
                header = r.fieldnames or []
                rows = list(r)
            self.keys = [k for k in header if k not in ("step", "epoch") and not k.endswith("_epoch")]
            keep = [row for row in rows if row.get("step") not in (None, "") and int(row["step"]) < int(start_step)]
            if len(keep) != len(rows) or header != self._header():
                self._rewrite(keep)
        else:
            self.path.parent.mkdir(parents=True, exist_ok=True)

    def _header(self):
        return ["step", "epoch"] + self.keys + [k + "_epoch" for k in self.keys]

    def _rewrite(self, rows):
        with open(self.path, "w", newline="") as f:
            w = csv.DictWriter(f, fieldnames=self._header(), restval="")
            w.writeheader()
            w.writerows(rows)

    def write(self, rows):
        """rows: dicts of step, epoch and key (or `<key>_epoch`) -> value."""
        if not rows:
            return
        new = [k for row in rows for k in row if k not in ("step", "epoch") and not k.endswith("_epoch")]
        new += [k[:-len("_epoch")] for row in rows for k in row if k.endswith("_epoch")]
        if [k for k in new if k not in self.keys] or not self.path.is_file():
            old = []
            if self.path.is_file():
                with open(self.path, newline="") as f:
                    old = list(csv.DictReader(f))
            assign_columns(self.keys, new)
            self._rewrite(old + [self._fmt(r) for r in rows])
            return
        with open(self.path, "a", newline="") as f:
            csv.DictWriter(f, fieldnames=self._header(), restval="").writerows([self._fmt(r) for r in rows])

    @staticmethod
    def _fmt(row):
        return {k: (v if k in ("step", "epoch") else repr(float(v))) for k, v in row.items()}


def logging_rows(keys, steps, epochs, values, every):
    """The CSV rows of a read-back block: the steps s with (s + 1) % every == 0, as Lightning's
    `log_every_n_steps` logs them.  Pure host function."""
    rows = []
    for j in np.flatnonzero((np.asarray(steps) + 1) % int(every) == 0):
        row = {"step": int(steps[j]), "epoch": int(epochs[j])}
        row.update({k: float(values[j, i]) for i, k in enumerate(keys)})
        rows.append(row)
    return rows


class TrainMetricsRecorder:
    """Every training step's logged `train/*` scalars, recorded on the device with no host sync (DESIGN.md section 15).

    `record(logged)` runs inside the step (and so inside its CUDA graph): one launch of tacorl_metrics_record writes the
    step's values to row (counter % ring_rows) of a ring_rows x 32 fp32 ring, adds each to an fp64 sum and a per-key
    count and advances the device counter.  Columns are the `train/*` keys in order of first appearance (at most 32); a
    key a later mode adds takes the next column and a key the step did not log is NaN in its row.  A plain Python
    number logged under `train/` is not recorded: it is a host value a captured graph would freeze.

    `step_done(global_step, epoch)` runs on the host after each step.  When a half of the ring fills, the rows are
    all-reduced to their mean over ranks on the training stream (between replays, in the same order on every rank), a
    side stream copies them to a pinned buffer, and the training stream waits for the previous copy out of the other
    half before it writes that half again.  Copies are read on the host at the next read-back, or by `flush()` (epoch and
    fit end), into `history` and, when given, `csv`.  `end_epoch()` also returns the epoch means from the rank-summed
    sums and counts.  `preserve()` lists the device state a step changes, so the warm-up steps of a capture record
    nothing."""

    def __init__(self, device, ring_rows, world=1, history=None, csv=None, log_every_n_steps=None):
        from . import _lib
        if int(ring_rows) < 2 or int(ring_rows) % 2:
            raise ValueError(f"ring_rows must be an even number >= 2, got {ring_rows}")
        device = torch.device(device)
        self.device = device if device.index is not None else torch.device("cuda", torch.cuda.current_device())
        self.ring_rows, self.half = int(ring_rows), int(ring_rows) // 2
        self.world = int(world)
        self.keys = []
        M = _lib.METRICS_MAX
        self.ring = torch.full((self.ring_rows, M), float("nan"), dtype=torch.float32, device=self.device)
        self.acc = torch.zeros(2 * M, dtype=torch.float64, device=self.device)
        self.counter = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.pinned = [torch.empty((self.half, M), dtype=torch.float32, pin_memory=True) for _ in range(2)]
        self.side = torch.cuda.Stream(device=self.device)
        self._filled = [torch.cuda.Event() for _ in range(2)]
        self._copied = [torch.cuda.Event() for _ in range(2)]
        self._queue = []         # copies not read yet, oldest first: (half, first row in the half, steps, epochs, keys)
        self.book = RingBook(self.half)
        self.history = history if history is not None else TrainHistory()
        self.csv = csv
        self.every = int(log_every_n_steps or self.half)
        self._hold = []

    def record(self, logged):
        from . import _lib
        names = [k for k, v in logged.items() if k.startswith("train/") and torch.is_tensor(v)]
        assign_columns(self.keys, names)
        m = _lib.Metrics()
        hold = []
        for k in names:
            v = logged[k]
            if v.numel() != 1 or v.device != self.device:
                raise ValueError(f"{k}: expected a one-element tensor on {self.device}, got {v!r}")
            if v.dtype != torch.float32 or not v.is_contiguous():
                v = v.float().contiguous()
                hold.append(v)           # keeps the converted value alive while the launch reads it
            m.value[self.keys.index(k)] = v.data_ptr()
        m.k, m.n = len(self.keys), 1
        self._hold = hold
        _lib.call("tacorl_metrics_record", ctypes.byref(m), _lib.ptr(self.ring), self.ring_rows,
                  _lib.ptr_any(self.counter), _lib.ptr_any(self.acc), _lib.stream())

    def preserve(self):
        return [self.counter, self.acc, self.ring]

    def step_done(self, global_step, epoch):
        got = self.book.advance(global_step, epoch)
        if got is not None:
            self._readback(got)

    def _readback(self, got):
        row0, steps, epochs = got
        h, off, n = row0 // self.half, row0 % self.half, len(steps)
        while any(q[0] == h for q in self._queue):       # the host has not read this half's previous copy yet
            self._read_oldest()
        main = torch.cuda.current_stream(self.device)
        rows = self.ring[row0:row0 + n]
        if self.world > 1:
            dist.all_reduce(rows)                        # training stream, between replays: every rank in one order
            rows.div_(self.world)
        self._filled[h].record(main)
        self.side.wait_event(self._filled[h])
        with torch.cuda.stream(self.side):
            self.pinned[h][off:off + n].copy_(rows, non_blocking=True)
            self._copied[h].record(self.side)
        self._queue.append((h, off, steps, epochs, list(self.keys)))
        main.wait_event(self._copied[1 - h])             # the training stream writes the other half next
        while self._queue and self._queue[0][0] != h and self._copied[self._queue[0][0]].query():
            self._read_oldest(wait=False)                # copies already done: read without waiting

    def _read_oldest(self, wait=True):
        h, off, steps, epochs, keys = self._queue.pop(0)
        if wait:
            self._copied[h].synchronize()
        vals = self.pinned[h][off:off + len(steps), :len(keys)].numpy().copy()
        self.history.append(keys, steps, epochs, vals)
        if self.csv is not None:
            self.csv.write(logging_rows(keys, steps, epochs, vals, self.every))

    def flush(self):
        """Reads everything recorded so far back to the host (waits for it)."""
        got = self.book.take()
        if got is not None:
            self._readback(got)
        while self._queue:
            self._read_oldest()

    def end_epoch(self):
        """flush(), then {key: epoch mean} from the sums and counts (summed over ranks), which are then zeroed."""
        self.flush()
        totals = self.acc.clone()
        if self.world > 1:
            dist.all_reduce(totals)
        means = epoch_means(self.keys, [totals.cpu().tolist()])
        self.acc.zero_()
        return means
