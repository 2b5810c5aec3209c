"""Launch-side drop-in for the part of `pl.Trainer` the reference's scripts/train.py:28-75 uses
(/root/reference/config/trainer/default.yaml:1-4: `strategy: ddp`, all GPUs, `precision: 16`; rl.yaml:4 `max_steps`):
one process per GPU (torchrun), NCCL gradient exchange through tacorl_b200.parallel instead of Lightning's DDP over
gloo, the whole optimisation step replayed from a CUDA graph, and checkpoints in Lightning's on-disk format (`epoch`,
`global_step`, `state_dict`, `optimizer_states`, `hyper_parameters`), so that runs resume from / are resumed by the
reference (`trainer.fit(model, ckpt_path=last.ckpt)`, train.py:48-66; utils/networks.py:90-117).

`B200Strategy` is the object to hand to a real `pl.Trainer(strategy=...)` when pytorch_lightning is installed; it is
only defined then.  This image has no pytorch_lightning, so `Trainer` below is what the tests and bench.py exercise."""
import os
from pathlib import Path

import torch
import torch.distributed as dist

from . import ops, parallel, runtime

CKPT_VERSION = "1.6.5"      # the reference pins pytorch-lightning < 1.7 (setup.cfg:17)
# the CUDA generator's seed during a validation sweep (restored afterwards): the same weights give the same metrics
VALIDATION_SEED = 0x7A11D


def _to_device(batch, device):
    return {k: (_to_device(v, device) if isinstance(v, dict) else (v.to(device) if torch.is_tensor(v) else v))
            for k, v in batch.items()}


def _optimizers_of(module):
    opts = module.optimizers() if hasattr(module, "optimizers") else module.configure_optimizers()
    return list(opts) if isinstance(opts, (list, tuple)) else [opts]


def save_checkpoint(module, path, epoch=0, global_step=0, extra=None):
    """Lightning-format checkpoint of a tacorl_b200 module (FlatAdam emits torch.optim.Adam's state layout)."""
    ckpt = {"epoch": int(epoch), "global_step": int(global_step), "pytorch-lightning_version": CKPT_VERSION,
            "state_dict": {k: v.detach().cpu().clone() for k, v in module.state_dict().items()},
            "optimizer_states": [o.state_dict() for o in _optimizers_of(module)],
            "lr_schedulers": [], "hyper_parameters": dict(getattr(module, "hparams", {}) or {})}
    if extra:
        ckpt.update(extra)
    path = Path(path)
    path.parent.mkdir(parents=True, exist_ok=True)
    torch.save(ckpt, path)
    return path


def restore_checkpoint(module, path, strict=True):
    """Loads weights, optimiser moments / step counts and the epoch counter from a Lightning-format checkpoint written
    by this package OR by the reference under Lightning (torch.optim.Adam states).  Returns the checkpoint dict."""
    ckpt = torch.load(path, map_location="cpu", weights_only=False)
    module.load_state_dict(ckpt["state_dict"], strict=strict)
    opts = _optimizers_of(module)
    states = ckpt.get("optimizer_states", [])
    assert len(states) in (0, len(opts)), f"checkpoint holds {len(states)} optimizer states, module has {len(opts)}"
    for o, s in zip(opts, states):
        o.load_state_dict(s)
        if hasattr(o, "invalidate_shadow"):
            o.invalidate_shadow()
    module.current_epoch = int(ckpt.get("epoch", 0))
    return ckpt


def _recording(step_fn, module, recorder):
    """step(batch), then the record launch of the `train/*` tensors that step logged.  A key whose tensor is the very
    object that was there before the step (`log` stores a new detached tensor each call) was not logged by it."""
    def step(batch):
        before = dict(module.logged)
        out = step_fn(batch)
        recorder.record({k: v for k, v in module.logged.items() if before.get(k) is not v})
        return out
    inner_preserve = step_fn.preserve
    step.mode_key = step_fn.mode_key
    step.preserve = lambda: list(inner_preserve()) + recorder.preserve()
    return step


class Trainer:
    """fit(module, batches) with the reference Trainer's knobs that matter on the hot path.
    batches: an iterable of batch dicts (host or device tensors), a callable step -> batch, or a DeviceReplay
    (tacorl_b200.replay: the batch is drawn and assembled on the device inside the step's graph); the loop runs one
    optimisation step per batch: `loss = training_step(batch, i); backward; optimizer.step()` for automatic optimisation
    (PlayLMP), `training_step(batch)` alone for manual optimisation (TACORL steps its own optimisers).
    Under torchrun (WORLD_SIZE > 1) every FlatAdam averages its gradient over the ranks (NCCL), overlapped with the
    encoder backward; rank r must be fed its own shard (parallel.shard_batch).

    Validation (`fit(..., val=)`, `validate`): every `check_val_every_n_epoch`-th epoch ends with a sweep of `val`, a
    DeviceReplay(mode="sweep") or a re-iterable of host batches, through the module's `validation_step`.  Each logged
    `validation/*` scalar becomes its item-weighted mean over the sweep (summed over ranks), in `callback_metrics` and
    `val_history`.  A sweep runs in eval mode under a fixed generator seed and leaves the training run untouched.

    Training metrics: every step's logged `train/*` tensors are recorded on the device inside the step (its CUDA graph
    included) and read back every `log_every_n_steps` steps without a host sync (runtime.TrainMetricsRecorder,
    DESIGN.md section 15).  `train_history` holds one row per step (mean over ranks), `train_epoch_metrics` the means of
    the last finished epoch and `train_epoch_history` one (epoch, global_step, means) entry per finished epoch; with
    `default_root_dir`, rank 0 also writes `metrics.csv`.  Python numbers logged under `train/` are not recorded."""

    def __init__(self, max_steps=-1, max_epochs=1, precision="bf16", use_cuda_graph=True, default_root_dir=None,
                 steps_per_epoch=None, save_every_n_epochs=1, device=None, check_val_every_n_epoch=1,
                 log_every_n_steps=50):
        self.max_steps, self.max_epochs = max_steps, max_epochs
        self.precision = {"16": "bf16", 16: "bf16", "bf16": "bf16", "32": "fp32", 32: "fp32", "fp32": "fp32"}[precision]
        self.use_cuda_graph = use_cuda_graph
        self.root = Path(default_root_dir) if default_root_dir else None
        self.steps_per_epoch = steps_per_epoch
        self.save_every_n_epochs = save_every_n_epochs
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.device = device or torch.device("cuda", self.local)
        self.global_step = 0
        self.losses = []
        if int(check_val_every_n_epoch) < 1:
            raise ValueError(f"check_val_every_n_epoch must be >= 1, got {check_val_every_n_epoch}")
        self.check_val_every_n_epoch = int(check_val_every_n_epoch)
        self.callback_metrics = {}
        self.val_history = []                 # (epoch, global_step, metrics) per sweep of fit()
        self._val_states = {}
        if int(log_every_n_steps) < 1:
            raise ValueError(f"log_every_n_steps must be >= 1, got {log_every_n_steps}")
        self.log_every_n_steps = int(log_every_n_steps)
        self.train_history = runtime.TrainHistory()
        self.train_epoch_metrics = {}
        self.train_epoch_history = []         # (epoch, global_step, {key: mean}) per finished epoch
        self._recorder = None
        self._train_graph = None

    def _setup_device(self, module):
        torch.cuda.set_device(self.device)
        ops.set_precision(self.precision)
        if self.world > 1 and not dist.is_initialized():
            os.environ.setdefault("NCCL_MAX_NCHANNELS", str(parallel.collective_channels(self.world)))
            os.environ.setdefault("NCCL_MIN_NCHANNELS", str(parallel.collective_channels(self.world)))
            dist.init_process_group("nccl", device_id=self.device)
        module.to(self.device)

    def _setup(self, module):
        self._setup_device(module)
        module.train()
        opts = _optimizers_of(module)
        if self.world > 1:
            for o in opts:
                parallel.attach_data_parallel(o, self.world)
        if getattr(module, "automatic_optimization", True):
            return runtime.play_lmp_step_fn(module, opts[0])
        return runtime.tacorl_step_fn(module)

    def fit(self, module, batches, ckpt_path=None, val=None):
        """batches: an iterable of batch dicts, a callable step -> batch, or a tacorl_b200.replay.DeviceReplay, which
        then samples every step's batch on the device (inside the step's CUDA graph).  With a replay, an epoch is
        `replay.steps_per_epoch` steps unless `steps_per_epoch` says otherwise, and checkpoints carry its step counter.
        val: validation data (see `validate`), swept at the end of every `check_val_every_n_epoch`-th epoch before
        that epoch's checkpoint is written; checkpoints then carry the results under "validation".
        Checkpoints carry the training epoch means under "training"; a resume restores them and appends to
        metrics.csv (dropping rows of steps at or after the checkpoint's)."""
        from .replay import DeviceReplay
        replay = batches if isinstance(batches, DeviceReplay) else None
        if replay is not None:
            if replay.mode != "train":
                raise ValueError("a sweep-mode DeviceReplay is a validation split: pass it as val=, not as the batches")
            self._check_replay(replay)
        if val is not None:
            self._check_val(val)
        step_fn = self._setup(module)
        if ckpt_path is not None and Path(ckpt_path).is_file():
            ckpt = restore_checkpoint(module, ckpt_path)
            self.global_step = int(ckpt.get("global_step", 0))
            if replay is not None and "replay" in ckpt:
                replay.load_state_dict(ckpt["replay"])
            if "validation" in ckpt:
                self.val_history = list(ckpt["validation"]["history"])
                self.callback_metrics = dict(ckpt["validation"]["metrics"])
            if "training" in ckpt:
                self.train_epoch_history = list(ckpt["training"]["epoch_history"])
                self.train_epoch_metrics = dict(ckpt["training"]["metrics"])
        rec = self._recorder = runtime.TrainMetricsRecorder(
            self.device, 2 * self.log_every_n_steps, world=self.world, history=self.train_history,
            csv=runtime.MetricsCSV(self.root / "metrics.csv", self.global_step) if self.root and self.rank == 0 else None,
            log_every_n_steps=self.log_every_n_steps)
        step_fn = _recording(step_fn, module, rec)
        if replay is not None:
            return self._fit_replay(module, step_fn, replay, val, rec)
        get = batches if callable(batches) else None
        it = None if get else iter(batches)
        graphed = None
        epoch0 = int(getattr(module, "current_epoch", 0))
        done_in_epoch = 0
        while True:
            if self.max_steps >= 0 and self.global_step >= self.max_steps:
                break
            if module.current_epoch - epoch0 >= self.max_epochs and self.max_steps < 0:
                break
            try:
                batch = get(self.global_step) if get else next(it)
            except StopIteration:
                break
            if batch is None:
                break
            if self.use_cuda_graph:
                if graphed is None:
                    graphed = self._train_graph = runtime.GraphedTrainStep(step_fn, batch, device=self.device, warmup=2)
                out = graphed(batch)
            else:
                out = step_fn(_to_device(batch, self.device))
            if torch.is_tensor(out):
                self.losses.append(out.detach().clone())
            rec.step_done(self.global_step, module.current_epoch)
            self.global_step += 1
            done_in_epoch += 1
            if self.steps_per_epoch and done_in_epoch >= self.steps_per_epoch:
                done_in_epoch = 0
                self._train_epoch_end(module, rec)
                self._end_of_epoch(module, val)
                module.current_epoch += 1          # (a graph captured for the BC epochs is swapped when bc_epochs is crossed)
                if self.root and self.rank == 0 and module.current_epoch % self.save_every_n_epochs == 0:
                    save_checkpoint(module, self.root / "saved_models" / f"tacorl_epoch_{module.current_epoch:02d}_.ckpt",
                                    module.current_epoch, self.global_step, extra=self._ckpt_extra(val))
        rec.flush()
        if self.root and self.rank == 0:
            save_checkpoint(module, self.root / "saved_models" / "last.ckpt", module.current_epoch, self.global_step,
                            extra=self._ckpt_extra(val))
        torch.cuda.synchronize(self.device)
        return self

    def _check_replay(self, replay):
        """A replay feeds the rank whose device holds it, with that rank's shard and random stream."""
        if torch.device(replay.device) != torch.device(self.device):
            raise ValueError(f"the replay lives on {replay.device} but this rank trains on {self.device}: build it with "
                             "device=cuda:LOCAL_RANK (the default under torchrun)")
        ix = replay.index
        if (ix.rank, ix.world_size) != (self.rank, self.world):
            raise ValueError(f"the replay holds shard {ix.rank} of {ix.world_size} but this is rank {self.rank} of "
                             f"{self.world}: build its ReplayIndex with rank=RANK, world_size=WORLD_SIZE")

    def _check_val(self, val):
        from .replay import DeviceReplay
        if isinstance(val, DeviceReplay):
            if val.mode != "sweep":
                raise ValueError("val= takes a DeviceReplay built with mode='sweep' (or an iterable of batches)")
            self._check_replay(val)
        elif callable(val) or not hasattr(val, "__iter__"):
            raise ValueError("val= takes a sweep-mode DeviceReplay or a re-iterable of batch dicts")

    def _ckpt_extra(self, val):
        extra = {"training": {"metrics": dict(self.train_epoch_metrics), "epoch_history": list(self.train_epoch_history)}}
        if val is not None:
            extra["validation"] = {"metrics": dict(self.callback_metrics), "history": list(self.val_history)}
        return extra

    def _train_epoch_end(self, module, rec):
        """The finished epoch's means of every recorded `train/*` key (rank-summed sums over rank-summed counts)."""
        means = rec.end_epoch()
        self.train_epoch_metrics = means
        self.train_epoch_history.append((int(module.current_epoch), int(self.global_step), dict(means)))
        if rec.csv is not None and means:
            row = {"step": self.global_step - 1, "epoch": int(module.current_epoch)}
            row.update({k + "_epoch": v for k, v in means.items()})
            rec.csv.write([row])

    def _end_of_epoch(self, module, val):
        """Lightning's rule: validate after epoch e when (e + 1) % check_val_every_n_epoch == 0 (current_epoch = e)."""
        if val is None or (module.current_epoch + 1) % self.check_val_every_n_epoch:
            return
        metrics = self._sweep(module, val)
        self.callback_metrics = dict(metrics)
        self.val_history.append((int(module.current_epoch), int(self.global_step), dict(metrics)))

    def validate(self, module, val):
        """One validation sweep of `module` over `val`: a DeviceReplay(mode="sweep") of this rank's split (full batches
        replayed from one CUDA graph, the tail run eagerly on prefix views) or a re-iterable of batch dicts (copied to
        the device, run eagerly).  Returns [{"validation/...": item-weighted mean}] like pl.Trainer.validate."""
        self._check_val(val)
        self._setup_device(module)
        metrics = self._sweep(module, val)
        self.callback_metrics = dict(metrics)
        return [metrics]

    def _sweep(self, module, val):
        """eval mode, the generator saved and seeded with VALIDATION_SEED, cursor and sums reset, every batch through
        validation_step_fn, one read-back of the (sums, count) vector (all-reduced over ranks first), then the
        generator and every submodule's train/eval flag restored."""
        from .replay import DeviceReplay
        key = (id(module), id(val))
        if key not in self._val_states:
            acc = runtime.MetricsAccumulator(self.device)
            self._val_states[key] = {"acc": acc, "step": runtime.validation_step_fn(module, acc), "graph": None}
        st = self._val_states[key]
        acc, step_fn = st["acc"], st["step"]
        flags = [(m, m.training) for m in module.modules()]
        with torch.cuda.device(self.device):
            rng = torch.cuda.get_rng_state()
            module.eval()
            try:
                if isinstance(val, DeviceReplay):
                    graphed = None
                    if self.use_cuda_graph and val.batches_per_sweep:
                        graphed = st["graph"]
                        if graphed is None:
                            graphed = st["graph"] = runtime.GraphedTrainStep(step_fn, None, device=self.device,
                                                                             warmup=2, source=val)
                        elif (graphed._key(), graphed._cur) != graphed._active_key:
                            graphed._select(graphed._key())     # capture a new host mode now, before the seed is set
                    torch.cuda.manual_seed(VALIDATION_SEED)
                    acc.reset()
                    val.reset()
                    for _ in range(val.batches_per_sweep):
                        if graphed is not None:
                            graphed()
                        else:
                            step_fn(val.sample())
                    if val.tail:
                        step_fn(val.sample(val.tail))
                else:
                    torch.cuda.manual_seed(VALIDATION_SEED)
                    acc.reset()
                    for batch in val:
                        step_fn(_to_device(batch, self.device))
                totals = acc.totals()
                if self.world > 1:
                    totals = totals.clone()
                    dist.all_reduce(totals)
                return acc.read(totals)
            finally:
                torch.cuda.set_rng_state(rng)
                for m, training in flags:
                    m.training = training

    def _fit_replay(self, module, step_fn, replay, val, rec):
        spe = self.steps_per_epoch or replay.steps_per_epoch
        graphed = None
        epoch0 = int(getattr(module, "current_epoch", 0))
        done_in_epoch = 0

        def save(name):
            if self.root and self.rank == 0:
                extra = {"replay": replay.state_dict()}
                extra.update(self._ckpt_extra(val))
                save_checkpoint(module, self.root / "saved_models" / name, module.current_epoch, self.global_step,
                                extra=extra)
        while not (self.max_steps >= 0 and self.global_step >= self.max_steps):
            if self.max_steps < 0 and module.current_epoch - epoch0 >= self.max_epochs:
                break
            if self.use_cuda_graph:
                if graphed is None:
                    graphed = self._train_graph = runtime.GraphedTrainStep(step_fn, None, device=self.device, warmup=2,
                                                                           source=replay)
                out = graphed()
            else:
                out = step_fn(replay.sample())
            if torch.is_tensor(out):
                self.losses.append(out.detach().clone())
            rec.step_done(self.global_step, module.current_epoch)
            self.global_step += 1
            done_in_epoch += 1
            if done_in_epoch >= spe:
                done_in_epoch = 0
                self._train_epoch_end(module, rec)
                self._end_of_epoch(module, val)
                module.current_epoch += 1
                if module.current_epoch % self.save_every_n_epochs == 0:
                    save(f"tacorl_epoch_{module.current_epoch:02d}_.ckpt")
        rec.flush()
        save("last.ckpt")
        torch.cuda.synchronize(self.device)
        return self


try:  # pragma: no cover - pytorch_lightning is not in this image
    import pytorch_lightning as pl

    class B200Strategy(pl.strategies.SingleDeviceStrategy):
        """`pl.Trainer(strategy=B200Strategy(), devices=1, ...)` per torchrun rank: Lightning keeps its loops, logging and
        checkpoint callbacks; the gradient exchange is tacorl_b200.parallel's NCCL all-reduce inside FlatAdam.step()."""

        def __init__(self):
            local = int(os.environ.get("LOCAL_RANK", "0"))
            super().__init__(device=torch.device("cuda", local))
            self._world = int(os.environ.get("WORLD_SIZE", "1"))

        def setup(self, trainer):
            if self._world > 1 and not dist.is_initialized():
                dist.init_process_group("nccl", device_id=self.root_device)
            super().setup(trainer)
            if self._world > 1:
                for o in trainer.optimizers:
                    parallel.attach_data_parallel(o, self._world)
except Exception:
    B200Strategy = None
