"""Train from an HBM-resident dataset: the frames are uploaded once, and every training step samples and assembles its own
batch on the device (tacorl_b200/csrc/replay.cu), inside the same CUDA graph as the optimisation step.  No frame
crosses PCIe after start-up.

    index = ReplayIndex.from_calvin("task_D_D/training", modalities=("rgb_static", "rgb_gripper"))
    replay = DeviceReplay(index, batch_size=64, kind="play_lmp", min_window=8, max_window=16, pad=6, seed=0)
    Trainer(max_steps=100_000).fit(module, replay)

`ReplayIndex` is host-only numpy: the rank's episodes as CHW uint8 frame arrays, the action rows, `ep_end[f]` (last
frame of f's episode) and the lookup tables the sampler draws from.  `DeviceReplay` holds the store on one device and
fills persistent output buffers in place; `sample()` returns the batch dict the modules consume (oracle/synth.py layout).
The sampling rules are DESIGN.md section 13: i.i.d. with replacement at every step, reproducible bit for bit from
(seed, rank, step).

`DeviceReplay(..., mode="sweep")` holds a validation split instead: every sweep visits each item of the rank's store
once, in store order, with per-item draws that depend on (seed, rank, item) only (DESIGN.md section 14).

    val = DeviceReplay(ReplayIndex.from_calvin("task_D_D/validation", ...), batch_size=64, kind="play_lmp",
                       min_window=8, max_window=16, seed=0, mode="sweep")
    Trainer(max_epochs=30).fit(module, replay, val=val)"""
import ctypes
import os

import numpy as np
import torch

from . import _lib as L

KINDS = {"play_lmp": 0, "tacorl": 1, "cql": 2}
UPLOAD_CHUNK_BYTES = 256 << 20


def geometric_thresholds(p, max_len=4096):
    """Inverse-CDF table of Geometric(p) on {1, 2, ...}: thr[k] = floor(2^32 P(d <= k + 1)), cut where it saturates.
    The device draws d = 1 + #{k : thr[k] <= u} for a uniform uint32 u: integer work only, no floating-point log."""
    if not 0.0 < p <= 1.0:
        raise ValueError(f"goal_p must be in (0, 1], got {p}")
    k = np.arange(1, max_len + 1, dtype=np.float64)
    with np.errstate(divide="ignore"):                  # p = 1: log1p(-1) = -inf, every threshold saturates
        decay = np.expm1(k * np.log1p(-p))
    thr = np.minimum(np.floor(np.ldexp(-decay, 32)), 2.0 ** 32 - 1)
    if thr[-1] < 2.0 ** 32 - 1:
        raise ValueError(f"Geometric({p}) keeps {float(decay[-1] + 1):.2e} of its mass beyond d = {max_len}: the "
                         f"{max_len}-entry table would cut the law off; use a larger goal_p")
    n = int(np.searchsorted(thr, 2.0 ** 32 - 1)) + 1
    return thr[:n].astype(np.uint32)


def shard_episodes(lengths, world_size):
    """Disjoint, size-balanced sets of whole episodes, one per rank: longest episode first onto the least-loaded rank.
    Loads then differ by at most one episode's length.  Returns a sorted list of episode positions per rank."""
    lengths = [int(n) for n in lengths]
    if world_size < 1 or len(lengths) < world_size:
        raise ValueError(f"{len(lengths)} episodes cannot be split over {world_size} ranks")
    load = [0] * world_size
    shards = [[] for _ in range(world_size)]
    for e in sorted(range(len(lengths)), key=lambda e: (-lengths[e], e)):
        r = min(range(world_size), key=lambda r: (load[r], r))
        shards[r].append(e)
        load[r] += lengths[e]
    return [sorted(s) for s in shards]


def _resize_hw(size):
    return (int(size), int(size)) if np.isscalar(size) else (int(size[0]), int(size[1]))


class ReplayIndex:
    """The rank's share of a dataset, laid out for the device store.

    episodes: list of dicts, one per episode, of arrays with the frame axis first: `rgb_*` HWC uint8 (n, H, W, 3) and
    the action key (n, A).  Under data parallelism pass every episode and `rank` / `world_size`: the rank keeps a
    size-balanced, disjoint set of whole episodes (shard_episodes).  resize: {modality: size or (h, w)}, applied once at
    load with torchvision's antialiased resize (the simulation pipeline's 200 -> 128 static frames)."""

    def __init__(self, episodes, modalities=("rgb_static",), action_key="rel_actions", resize=None, rank=0,
                 world_size=1, episode_ids=None):
        self.modalities = tuple(modalities)
        self.action_key = action_key
        self.rank, self.world_size = int(rank), int(world_size)
        ids = list(range(len(episodes))) if episode_ids is None else list(episode_ids)
        mine = shard_episodes([len(ep[action_key]) for ep in episodes], self.world_size)[self.rank]
        self._build([episodes[e] for e in mine], [ids[e] for e in mine], resize or {})

    @classmethod
    def from_calvin(cls, root, modalities=("rgb_static",), action_key="rel_actions", resize=None, rank=0, world_size=1):
        """CALVIN layout: `ep_start_end_ids.npy` with inclusive [start, end] frame ids per episode and one
        `episode_{id:07d}.npz` per frame.  Only this rank's episodes are read."""
        bounds = np.asarray(np.load(os.path.join(root, "ep_start_end_ids.npy")), dtype=np.int64).reshape(-1, 2)
        bounds = bounds[np.argsort(bounds[:, 0], kind="stable")]
        if (bounds[:, 1] < bounds[:, 0]).any():
            raise ValueError(f"{root}: an episode ends before it starts")
        mine = shard_episodes(bounds[:, 1] - bounds[:, 0] + 1, world_size)[rank]
        self = cls.__new__(cls)
        self.modalities, self.action_key = tuple(modalities), action_key
        self.rank, self.world_size = int(rank), int(world_size)
        keys = list(self.modalities) + [action_key]
        episodes = []
        for e in mine:
            lo, hi = int(bounds[e, 0]), int(bounds[e, 1])
            frames = {k: [] for k in keys}
            for i in range(lo, hi + 1):
                with np.load(os.path.join(root, f"episode_{i:07d}.npz")) as f:     # one open file at a time
                    for k in keys:
                        frames[k].append(f[k])
            episodes.append({k: np.stack(v) for k, v in frames.items()})
        self._build(episodes, [int(bounds[e, 0]) for e in mine], resize or {})
        return self

    def _build(self, episodes, ids, resize):
        if not episodes:
            raise ValueError("no episode on this rank")
        self.episode_ids = list(ids)
        lengths = np.array([len(ep[self.action_key]) for ep in episodes], dtype=np.int64)
        if (lengths < 1).any():
            raise ValueError("empty episode")
        self.frames = {}
        for m in self.modalities:
            chw = []
            for ep in episodes:
                x = np.asarray(ep[m])
                if x.dtype != np.uint8 or x.ndim != 4 or x.shape[-1] != 3:
                    raise ValueError(f"{m}: expected HWC uint8 frames (n, H, W, 3), got {x.dtype} {x.shape}")
                x = np.ascontiguousarray(x.transpose(0, 3, 1, 2))
                if m in resize:
                    import torchvision.transforms.functional as TF
                    x = TF.resize(torch.from_numpy(x), list(_resize_hw(resize[m])), antialias=True).numpy()
                chw.append(x)
            self.frames[m] = np.ascontiguousarray(np.concatenate(chw))
            if self.frames[m].shape[-1] % 4:
                raise ValueError(f"{m}: frame width {self.frames[m].shape[-1]} is not a multiple of 4")
        self.actions = np.ascontiguousarray(np.concatenate([np.asarray(ep[self.action_key], np.float32)
                                                            for ep in episodes]))
        ends = np.cumsum(lengths) - 1
        self.ep_end = np.repeat(ends, lengths).astype(np.int32)
        self.episode_lengths = lengths
        if len(self.ep_end) >= 2 ** 31 - 1:
            raise ValueError("more than 2^31 frames on one rank")

    @property
    def num_frames(self):
        return len(self.ep_end)

    def valid_starts(self, min_window):
        """Window starts: frames with at least `min_window` frames left in their episode."""
        f = np.arange(self.num_frames, dtype=np.int64)
        return np.nonzero(self.ep_end - f + 1 >= int(min_window))[0].astype(np.int32)

    def valid_transitions(self):
        """Transition starts: frames with a successor in their episode."""
        return np.nonzero(self.ep_end > np.arange(self.num_frames))[0].astype(np.int32)

    def items(self, kind, min_window=1):
        """The start table a replay of `kind` draws from, and a sweep visits in order: window starts (play_lmp,
        tacorl) or transition starts (cql)."""
        return self.valid_transitions() if kind == "cql" else self.valid_starts(min_window)

    def geometric_thresholds(self, p):
        return geometric_thresholds(p)

    @property
    def nbytes(self):
        """Bytes of the device store: frames, action rows and ep_end (the lookup tables come on top)."""
        return sum(a.nbytes for a in self.frames.values()) + self.actions.nbytes + self.ep_end.nbytes


def _jitter_params(jitter):
    """jitter dict -> {"c": tacorl_replay_jitter, "mean", "std", "ranges"} or None (no op enabled)."""
    if jitter is None:
        return None
    unknown = set(jitter) - {"brightness", "contrast", "hue", "mean", "std"}
    if unknown:
        raise ValueError(f"unknown jitter keys {sorted(unknown)}")
    b, c, h = (float(jitter.get(k, 0.0)) for k in ("brightness", "contrast", "hue"))
    if min(b, c, h) < 0 or h > 0.5:
        raise ValueError(f"jitter strengths must be >= 0 (hue <= 0.5), got {b}, {c}, {h}")
    if not (b or c or h):
        return None
    ranges = [(max(0.0, 1 - b), 1 + b), (max(0.0, 1 - c), 1 + c), (-h, h)]
    cs = L.ReplayJitter()
    cs.ops = (1 if b else 0) | (2 if c else 0) | (8 if h else 0)
    for i, (lo, hi) in enumerate(ranges):      # float32 lo and span: the device and the oracle use these values
        cs.lo[i] = float(np.float32(lo))
        cs.span[i] = float(np.float32(hi) - np.float32(lo))
    std = float(jitter.get("std", 0.5))
    if std == 0:
        raise ValueError("jitter std must not be zero")
    return {"c": cs, "mean": float(jitter.get("mean", 0.5)), "std": std, "ops": cs.ops,
            "lo": [cs.lo[i] for i in range(3)], "span": [cs.span[i] for i in range(3)]}


def sweep_shape(items, batch_size):
    """(full batches, tail rows) of a sweep over `items` items: every item once, the tail neither padded nor dropped."""
    return int(items) // int(batch_size), int(items) % int(batch_size)


def _prefix(batch, n):
    return {k: (_prefix(v, n) if isinstance(v, dict) else v[:n]) for k, v in batch.items()}


def _validate(index, valid):
    F = index.num_frames
    f = np.arange(F)
    if not ((index.ep_end >= f) & (index.ep_end < F)).all():
        raise ValueError("ep_end holds a frame id outside its episode or the store")
    if len(valid) == 0:
        raise ValueError("no valid start on this rank (episodes shorter than the minimum window?)")
    if valid.min() < 0 or valid.max() >= F:
        raise ValueError("start table holds an out-of-range frame id")


class DeviceReplay:
    """HBM-resident replay of one rank.  `sample()` draws the next step's batch and assembles it in persistent buffers
    (stable addresses: the call may be captured in a CUDA graph) and returns the batch dict:
      play_lmp  states{m} (B, T, 3, H, W), actions (B, T, A), idx, window_size (B,) int64;
      tacorl    the same plus goal{m} (B, 3, H, W) and disp (B,) int64 (-1 for a negative goal);
      cql       observations{observation{m}, goal{m}}, actions (B, A), next_observations{observation{m}, goal{m}},
                rewards, terminals (B,) int64.
    Frames are uint8 (the encoders normalise them on load).  T = max_window; pad > 0 applies RandomShiftsAug(pad) to
    every frame with its own shift.  jitter = {"brightness": b, "contrast": c, "hue": h[, "mean": 0.5, "std": 0.5]}:
    ColorTransform of rl_train.yaml on every frame with its own op order and factors (torchvision ColorJitter ranges
    [max(0, 1 - b), 1 + b], [max(0, 1 - c), 1 + c], [-h, h]), then Normalize(mean, std): frames come out float32.
    The step counter lives on the device and advances inside sample().  device defaults to cuda:LOCAL_RANK under
    torchrun (else the current device); sample() always launches on that device's current stream.

    mode="sweep": a validation split.  The items (window starts; CQL: transitions) form `batches_per_sweep` full
    batches and a `tail` of `items % batch_size` rows; `reset()` puts the device item cursor at 0 and `sample(n)` fills
    rows [0, n) from the next n items and returns prefix views.  No augmentation: pad must be 0 and jitter None."""

    def __init__(self, index, batch_size, kind="play_lmp", min_window=8, max_window=16, pad=0, goal_p=0.3,
                 neg_frac=0.1, jitter=None, seed=0, device=None, mode="train"):
        if kind not in KINDS:
            raise ValueError(f"kind must be one of {sorted(KINDS)}, got {kind!r}")
        if mode not in ("train", "sweep"):
            raise ValueError(f"mode must be 'train' or 'sweep', got {mode!r}")
        if mode == "sweep" and (int(pad) > 0 or _jitter_params(jitter) is not None):
            raise ValueError("a validation sweep does not augment: build it with pad=0 and jitter=None")
        self.mode = mode
        if kind != "cql" and not 1 <= min_window <= max_window:
            raise ValueError(f"window bounds {min_window}..{max_window}")
        if not 0.0 <= neg_frac <= 1.0:
            raise ValueError(f"neg_frac must be in [0, 1], got {neg_frac}")
        self.index, self.kind, self.B = index, kind, int(batch_size)
        self.min_window, self.max_window = int(min_window), int(max_window)
        self.T = 1 if kind == "cql" else self.max_window
        self.pad, self.goal_p, self.neg_frac = int(pad), float(goal_p), float(neg_frac)
        self.seed, self.rank = int(seed), int(index.rank)
        if device is None:
            local = os.environ.get("LOCAL_RANK")
            device = torch.device("cuda", int(local) if local is not None else torch.cuda.current_device())
        device = torch.device(device)
        if device.type != "cuda":
            raise ValueError(f"DeviceReplay needs a CUDA device, got {device}")
        self.device = device if device.index is not None else torch.device("cuda", torch.cuda.current_device())
        self.jitter = _jitter_params(jitter)
        mods = index.modalities
        self.n_slots = {"play_lmp": self.T, "tacorl": self.T + 1, "cql": 3}[kind]
        valid = index.items(kind, self.min_window)
        # goals and CQL offsets draw from the geometric table; PlayLMP never reads it
        geom = geometric_thresholds(self.goal_p) if kind != "play_lmp" else np.full(1, 2 ** 32 - 1, np.uint32)
        _validate(index, valid)
        B, T = self.B, self.T
        per_sample = sum(3 * a.shape[2] * a.shape[3] for a in index.frames.values())
        out_frames = {"play_lmp": T, "tacorl": T + 1, "cql": 3}[kind]
        A = index.actions.shape[1]
        self.output_bytes = B * (out_frames * per_sample + (T if kind != "cql" else 1) * A * 4 + 3 * 8 + 4 * 4)
        if self.pad > 0:
            self.output_bytes += len(mods) * B * self.n_slots * 2 * 4
        if self.jitter is not None:       # float32 frames + op order, factors and contrast means per frame
            self.output_bytes += B * out_frames * (4 * per_sample + len(mods) * 4 * 5)
        self.table_bytes = valid.nbytes + geom.nbytes + 8
        need = index.nbytes + self.table_bytes + self.output_bytes
        free, total = torch.cuda.mem_get_info(self.device)
        if need > free:
            raise MemoryError(f"DeviceReplay needs {need} bytes on {self.device} (store {index.nbytes}, tables "
                              f"{self.table_bytes}, batch buffers {self.output_bytes}) but only {free} of {total} are "
                              "free; split the episodes over more ranks (ReplayIndex(rank=, world_size=)) or resize")
        dev = self.device
        with torch.cuda.device(dev):
            self._allocate(index, valid, geom)

    def _allocate(self, index, valid, geom):
        dev, B, mods = self.device, self.B, index.modalities
        self.store = {m: self._upload(index.frames[m]) for m in mods}
        self.actions_store = self._upload(index.actions)
        self.ep_end = self._upload(index.ep_end)
        self.valid = self._upload(valid)
        self.n_valid = len(valid)
        self.geom = self._upload(geom.view(np.int32))
        self.n_geom = len(geom)
        # negative goal iff u < neg_thr over uint32 u: neg_frac = 1 gives 2^32, every draw
        self.neg_thr = int(np.floor(self.neg_frac * 2.0 ** 32)) if self.kind == "tacorl" else 0
        self._step = torch.zeros(1, dtype=torch.int64, device=dev)
        self.tab = torch.zeros(4, B, dtype=torch.int32, device=dev)
        self.out64 = torch.zeros(3, B, dtype=torch.int64, device=dev)
        self.shift = (torch.zeros(len(mods), B, self.n_slots, 2, dtype=torch.int32, device=dev) if self.pad > 0
                      else None)
        self.jit_order = self.jit_factors = None
        if self.jitter is not None:
            self.jit_order = torch.zeros(len(mods), B, self.n_slots, dtype=torch.int32, device=dev)
            self.jit_factors = torch.zeros(len(mods), B, self.n_slots, 3, dtype=torch.float32, device=dev)
        self._alloc_outputs()

    def _upload(self, arr):
        """Host array -> device tensor with ordinary copies, in chunks of about UPLOAD_CHUNK_BYTES."""
        src = torch.from_numpy(np.ascontiguousarray(arr))
        dst = torch.empty(src.shape, dtype=src.dtype, device=self.device)
        rows = max(1, UPLOAD_CHUNK_BYTES // max(1, src[:1].numel() * src.element_size()))
        for i in range(0, src.shape[0], rows):
            dst[i:i + rows].copy_(src[i:i + rows])
        return dst

    def _alloc_outputs(self):
        B, T, dev = self.B, self.T, self.device
        A = self.index.actions.shape[1]

        def img(m, nf):
            _, c, h, w = self.index.frames[m].shape
            shape = (B, nf, c, h, w) if nf else (B, c, h, w)
            return torch.empty(shape, dtype=torch.uint8, device=dev)

        mods = self.index.modalities
        jobs = []           # (modality, role, shift slot, output dict)
        if self.kind == "cql":
            self.obs, self.next_obs, self.goal = {}, {}, {}
            for m in mods:
                jobs += [(m, L.REPLAY_OBS, 0, self.obs), (m, L.REPLAY_NEXT, 1, self.next_obs),
                         (m, L.REPLAY_GOAL, 2, self.goal)]
            self.actions = torch.empty(B, A, dtype=torch.float32, device=dev)
        else:
            self.states = {}
            jobs += [(m, L.REPLAY_WINDOW, 0, self.states) for m in mods]
            if self.kind == "tacorl":
                self.goal = {}
                jobs += [(m, L.REPLAY_GOAL, T, self.goal) for m in mods]
            self.actions = torch.empty(B, T, A, dtype=torch.float32, device=dev)
        # the gather writes uint8 frames; with jitter they are staging for the float32 frames the batch holds
        self._jit_jobs = []
        for i, (m, role, slot, d) in enumerate(jobs):
            nf = T if role == L.REPLAY_WINDOW else 0
            u8 = img(m, nf)
            if self.jitter is None:
                d[m] = u8
            else:
                d[m] = torch.empty(u8.shape, dtype=torch.float32, device=dev)
                ws = torch.empty(B * max(nf, 1), dtype=torch.float32, device=dev)
                self._jit_jobs.append((u8, d[m], mods.index(m), max(nf, 1), slot, ws))
            jobs[i] = (m, role, slot, u8)
        if len(jobs) > L.REPLAY_MAX_IMAGES:
            raise ValueError(f"{len(jobs)} image outputs; the gather takes at most {L.REPLAY_MAX_IMAGES}")
        self._images = (L.ReplayImage * max(1, len(jobs)))()
        for i, (m, role, slot, out) in enumerate(jobs):
            st = self.store[m]
            sh = None if self.shift is None else self.shift[mods.index(m)].data_ptr()
            self._images[i] = L.ReplayImage(st.data_ptr(), out.data_ptr(), sh, st.shape[2], st.shape[3], role, slot,
                                            self.n_slots)
        self._n_images = len(jobs)

    # ---- the step
    def sample(self, n=None):
        """Draw and assemble the next batch on the current stream (two launches); returns the batch dict.
        Sweep mode: rows [0, n) (default: the whole batch) from the next n items; the batch dict holds prefix views."""
        if self.mode == "sweep":
            return self._sweep(self.B if n is None else int(n))
        if n is not None:
            raise ValueError("a training replay always draws whole batches: call sample() without n")
        with torch.cuda.device(self.device):
            s = L.stream()
            jit = None if self.jitter is None else ctypes.byref(self.jitter["c"])
            L.call("tacorl_replay_sample", KINDS[self.kind], self.B, self.min_window, self.max_window,
                   len(self.index.modalities), self.n_slots, self.pad, self.neg_thr, self.seed & 0xFFFFFFFFFFFFFFFF,
                   self.rank, L.ptr_any(self._step), L.ptr_any(self.ep_end), self.index.num_frames,
                   L.ptr_any(self.valid), self.n_valid, L.ptr_any(self.geom), self.n_geom, L.ptr_any(self.tab),
                   L.ptr_any(self.shift), L.ptr_any(self.out64), jit, L.ptr_any(self.jit_order),
                   L.ptr_any(self.jit_factors), s)
            act_role = L.REPLAY_OBS if self.kind == "cql" else L.REPLAY_WINDOW
            L.call("tacorl_replay_gather", self.B, self.T, self.pad, L.ptr_any(self.tab), self._n_images,
                   ctypes.cast(self._images, ctypes.c_void_p), L.ptr_any(self.actions_store), self.actions.shape[-1],
                   act_role, 1 if self.action_zero_pad else 0, L.ptr_any(self.actions), s)
            for u8, out, mi, nf, slot, ws in self._jit_jobs:
                h, w = u8.shape[-2:]
                L.call("tacorl_replay_color_jitter", L.ptr_any(u8), self.B, nf, h, w, L.ptr_any(self.jit_order[mi]),
                       L.ptr(self.jit_factors[mi]), self.n_slots, slot, self.jitter["mean"], self.jitter["std"],
                       L.ptr(ws), L.ptr(out), s)
        return self.batch()

    def _sweep(self, n):
        if not 1 <= n <= self.B:
            raise ValueError(f"a sweep batch holds 1..{self.B} rows, got {n}")
        with torch.cuda.device(self.device):
            s = L.stream()
            L.call("tacorl_replay_sweep", KINDS[self.kind], self.B, n, self.min_window, self.max_window, self.neg_thr,
                   self.seed & 0xFFFFFFFFFFFFFFFF, self.rank, L.ptr_any(self._step), L.ptr_any(self.ep_end),
                   self.index.num_frames, L.ptr_any(self.valid), self.n_valid, L.ptr_any(self.geom), self.n_geom,
                   L.ptr_any(self.tab), L.ptr_any(self.out64), s)
            act_role = L.REPLAY_OBS if self.kind == "cql" else L.REPLAY_WINDOW
            L.call("tacorl_replay_gather_rows", self.B, n, self.T, 0, L.ptr_any(self.tab), self._n_images,
                   ctypes.cast(self._images, ctypes.c_void_p), L.ptr_any(self.actions_store), self.actions.shape[-1],
                   act_role, 1 if self.action_zero_pad else 0, L.ptr_any(self.actions), s)
        return self.batch(n)

    @property
    def action_zero_pad(self):
        """Relative actions pad with zeros (gripper repeated); absolute ones repeat the last step."""
        return self.index.action_key.startswith("rel")

    def batch(self, n=None):
        """The batch dict over the persistent buffers (a fresh dict each call: modules may rebind its entries).
        n: views of the first n rows only (a sweep's tail)."""
        if n is not None:
            full = self.batch()
            return _prefix(full, int(n))
        if self.kind == "cql":
            return {"observations": {"observation": dict(self.obs), "goal": dict(self.goal)}, "actions": self.actions,
                    "next_observations": {"observation": dict(self.next_obs), "goal": dict(self.goal)},
                    "rewards": self.out64[0], "terminals": self.out64[1]}
        out = {"states": dict(self.states), "actions": self.actions, "idx": self.out64[0], "window_size": self.out64[1]}
        if self.kind == "tacorl":
            out["goal"] = dict(self.goal)
            out["disp"] = self.out64[2]
        return out

    # ---- state
    @property
    def launches_per_sample(self):
        """Library launches of one sample(): sampler, gather, and two per jittered image output."""
        return 2 + 2 * len(self._jit_jobs)

    @property
    def step(self):
        """Steps drawn so far (reads the device counter: synchronises)."""
        return int(self._step.item())

    def preserve(self):
        """Tensors sample() mutates that a graph capture must restore (GraphedTrainStep): the step counter, or in
        sweep mode the item cursor."""
        return [self._step]

    # ---- sweep mode
    @property
    def items(self):
        """Items of one sweep: valid window starts (CQL: transitions) on this rank."""
        return self.n_valid

    @property
    def batches_per_sweep(self):
        """Full batches of one sweep."""
        return sweep_shape(self.n_valid, self.B)[0]

    @property
    def tail(self):
        """Rows of the sweep's last, partial batch (0: none)."""
        return sweep_shape(self.n_valid, self.B)[1]

    def reset(self):
        """Put the sweep's item cursor at the first item (on the device's current stream)."""
        if self.mode != "sweep":
            raise ValueError("reset() rewinds a validation sweep; a training replay resumes with load_state_dict()")
        with torch.cuda.device(self.device):
            self._step.zero_()

    @property
    def steps_per_epoch(self):
        """Valid starts on this rank divided by the per-rank batch (at least 1)."""
        return max(1, self.n_valid // self.B)

    def state_dict(self):
        return {"step": self.step, "seed": self.seed, "rank": self.rank}

    def load_state_dict(self, state):
        self._step.fill_(int(state["step"]))
