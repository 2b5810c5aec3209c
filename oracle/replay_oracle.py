"""TEST INFRASTRUCTURE — numpy restatement of the HBM-resident replay (tacorl_b200/csrc/replay.cu): the Philox4x32-10
draws, their integer mappings, and the batch assembly.  The sampling rules are DESIGN.md section 13.  The product package
never imports this module.

Window padding and action padding are the ones of transforms_oracle (pad_frames, pad_rel_actions); the shift is the
integer form of RandomShiftsAug.  `shift_frames` restates it with index clamping, so it also covers non-square frames.
tests/test_replay_host.py pins it to transforms_oracle.random_shifts on square frames."""
import numpy as np
import torch

from oracle import transforms_oracle as TO

PLAY_LMP, TACORL, CQL = 0, 1, 2
KINDS = {"play_lmp": PLAY_LMP, "tacorl": TACORL, "cql": CQL}
DRAW_SAMPLE, DRAW_NEG_GOAL, DRAW_SHIFT0 = 0, 1, 2
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox4x32-10 over broadcastable uint32 arrays.  Returns the four output words (uint32 arrays)."""
    c = [np.asarray(v, dtype=np.uint64) & _M32 for v in (c0, c1, c2, c3)]
    c = list(np.broadcast_arrays(*c))
    k0, k1 = np.uint64(k0) & _M32, np.uint64(k1) & _M32
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _M32
        hi1, lo1 = p1 >> np.uint64(32), p1 & _M32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(0x9E3779B9)) & _M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & _M32
    return [v.astype(np.uint32) for v in c]


def key(seed, rank):
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return seed & 0xFFFFFFFF, ((seed >> 32) ^ ((int(rank) * 0x9E3779B9) & 0xFFFFFFFF)) & 0xFFFFFFFF


def uniform_below(u, n):
    """(uint64(u) * n) >> 32."""
    return ((np.asarray(u, dtype=np.uint64) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)


def geometric_thresholds(p, max_len=4096):
    """thr[k] = floor(2^32 P(d <= k + 1)) for d ~ Geometric(p) on {1, 2, ...}; stops once the threshold saturates."""
    k = np.arange(1, max_len + 1, dtype=np.float64)
    with np.errstate(divide="ignore"):                  # p = 1: log1p(-1) = -inf, every threshold saturates
        decay = np.expm1(k * np.log1p(-p))
    thr = np.floor(np.ldexp(-decay, 32))
    thr = np.minimum(thr, 2.0 ** 32 - 1)
    n = int(np.searchsorted(thr, 2.0 ** 32 - 1)) + 1
    return thr[:min(n, max_len)].astype(np.uint32)


def geometric(u, thr):
    """1 + #{k : thr[k] <= u}."""
    return np.searchsorted(thr.astype(np.int64), np.asarray(u, dtype=np.int64), side="right") + 1


JITTER_PERMS = ((0, 1, 3), (0, 3, 1), (1, 0, 3), (1, 3, 0), (3, 0, 1), (3, 1, 0))


def uniform_float(u, lo, span):
    """lo + span * (u >> 8) * 2^-24 in float32, each operation rounded once (the device's __fmul_rn / __fadd_rn)."""
    x = (np.asarray(u, dtype=np.uint32) >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)
    return np.float32(lo) + np.float32(span) * x


def unpack_order(code):
    """Packed op order (4 bits per op, first op lowest, 0xF = none) -> list of op ids."""
    return [(int(code) >> (4 * k)) & 0xF for k in range(3) if ((int(code) >> (4 * k)) & 0xF) != 0xF]


def sample(kind, step, B, seed, rank, ep_end, valid, *, min_window=1, max_window=1, geom_thr=None, neg_thr=0,
           n_mod=0, n_slots=0, pad=0, jitter=None):
    """The tables replay_sample_kernel writes for one step: dict of int32 `tab` (4, B), int64 `out64` (3, B), int32
    `shift` (n_mod, B, n_slots, 2) or None, and with jitter = {"ops", "lo", "span"} int32 `jit_order` (n_mod, B,
    n_slots) and float32 `jit_factors` (n_mod, B, n_slots, 3)."""
    kind = KINDS.get(kind, kind)
    k0, k1 = key(seed, rank)
    c0, c1 = int(step) & 0xFFFFFFFF, (int(step) >> 32) & 0xFFFFFFFF
    b = np.arange(B, dtype=np.uint64)
    r = philox4x32_10(c0, c1, b, DRAW_SAMPLE, k0, k1)
    ep_end = np.asarray(ep_end, dtype=np.int64)
    valid = np.asarray(valid, dtype=np.int64)
    s = valid[uniform_below(r[0], len(valid))]
    end = ep_end[s]
    if kind == CQL:
        k = geometric(r[3], geom_thr)
        goal = np.minimum(s + k, end)
        hit = (goal == s + 1).astype(np.int64)
        tab = np.stack([s, np.ones(B, np.int64), goal, hit])
        out64 = np.stack([hit, hit, goal])
    else:
        wmax = np.minimum(max_window, end - s + 1)
        n_sizes = (wmax - min_window + 1).astype(np.uint64)
        w = min_window + ((r[1].astype(np.uint64) * n_sizes) >> np.uint64(32)).astype(np.int64)
        last = s + w - 1
        goal, disp = last.copy(), np.ones(B, np.int64)
        if kind == TACORL:
            neg = r[2].astype(np.int64) < int(neg_thr)
            g = philox4x32_10(c0, c1, b, DRAW_NEG_GOAL, k0, k1)
            d = geometric(r[3], geom_thr)
            pos_goal = np.minimum(last + d - 1, end)
            goal = np.where(neg, uniform_below(g[0], len(ep_end)), pos_goal)
            disp = np.where(neg, -1, goal - last + 1)
        tab = np.stack([s, w, goal, disp])
        out64 = np.stack([s, w, disp])
    shift = None
    jit_order = jit_factors = None
    if jitter is not None:
        m, bb, j = np.meshgrid(np.arange(n_mod), np.arange(B), np.arange(n_slots), indexing="ij")
        draw = DRAW_SHIFT0 + n_mod * n_slots + m * n_slots + j
        rj = philox4x32_10(c0, c1, bb.astype(np.uint64), draw.astype(np.uint64), k0, k1)
        perm = uniform_below(rj[0], 6)
        ops = int(jitter["ops"])
        jit_order = np.empty(perm.shape, np.int32)
        for idx, p in np.ndenumerate(perm):
            en = [o for o in JITTER_PERMS[p] if (ops >> o) & 1]
            en += [0xF] * (3 - len(en))
            jit_order[idx] = en[0] | (en[1] << 4) | (en[2] << 8)
        lo, span = jitter["lo"], jitter["span"]
        jit_factors = np.stack([uniform_float(rj[1], lo[0], span[0]) if ops & 1 else np.ones(perm.shape, np.float32),
                                uniform_float(rj[2], lo[1], span[1]) if ops & 2 else np.ones(perm.shape, np.float32),
                                uniform_float(rj[3], lo[2], span[2]) if ops & 8 else np.zeros(perm.shape, np.float32)],
                               -1).astype(np.float32)
    if n_mod and n_slots and pad is not None and pad > 0:
        m, bb, j = np.meshgrid(np.arange(n_mod), np.arange(B), np.arange(n_slots), indexing="ij")
        draw = DRAW_SHIFT0 + m * n_slots + j
        rs = philox4x32_10(c0, c1, bb.astype(np.uint64), draw.astype(np.uint64), k0, k1)
        shift = np.stack([uniform_below(rs[0], 2 * pad + 1), uniform_below(rs[1], 2 * pad + 1)], -1).astype(np.int32)
    return {"tab": tab.astype(np.int32), "out64": out64.astype(np.int64), "shift": shift, "jit_order": jit_order,
            "jit_factors": jit_factors}


def jitter_frames(u8, order, factors, mean=0.5, std=0.5):
    """ScaleImageTensor -> ColorJitter (transforms_oracle.color_jitter with the drawn order / factors) -> Normalize of
    uint8 frames (n, 3, h, w); order (n,), factors (n, 3).  float32 torch tensor."""
    x = TO.scale_image(torch.as_tensor(np.asarray(u8)))
    out = [TO.normalize(TO.color_jitter(x[i], unpack_order(order[i]), float(factors[i][0]), float(factors[i][1]),
                                        float(factors[i][2])), mean, std) for i in range(x.shape[0])]
    return torch.stack(out)


def shift_frames(x, shift, pad):
    """Integer RandomShiftsAug: x uint8 (n, c, h, w), shift (n, 2) in [0, 2 pad] (x then y): out[y][x] =
    x[clamp(y + sy - pad)][clamp(x + sx - pad)]."""
    x = np.asarray(x)
    n, _, h, w = x.shape
    out = np.empty_like(x)
    for i in range(n):
        ys = np.clip(np.arange(h) + int(shift[i][1]) - pad, 0, h - 1)
        xs = np.clip(np.arange(w) + int(shift[i][0]) - pad, 0, w - 1)
        out[i] = x[i][:, ys][:, :, xs]
    return out


def assemble(kind, tables, frames, actions, T, pad, modalities, zero_pad=True):
    """The batch replay_gather_kernel writes from `tables` (see `sample`): frames {m: uint8 (F, 3, H, W)}, actions
    float32 (F, A).  Returns the batch dict (torch tensors) with the keys DeviceReplay.sample() returns."""
    kind = KINDS.get(kind, kind)
    tab, out64, shift = tables["tab"], tables["out64"], tables["shift"]
    B = tab.shape[1]
    s, w, goal = tab[0].astype(np.int64), tab[1].astype(np.int64), tab[2].astype(np.int64)

    def shifted(m, imgs, slot0):
        if shift is None:
            return imgs
        mi = modalities.index(m)
        return np.stack([shift_frames(imgs[b], shift[mi, b, slot0:slot0 + imgs.shape[1]], pad) for b in range(B)])

    def single(m, ids, slot):
        return torch.from_numpy(shifted(m, frames[m][ids][:, None], slot)[:, 0].copy())

    acts = torch.from_numpy(np.asarray(actions))
    if kind == CQL:
        obs = {m: single(m, s, 0) for m in modalities}
        nxt = {m: single(m, s + 1, 1) for m in modalities}
        gl = {m: single(m, goal, 2) for m in modalities}
        return {"observations": {"observation": obs, "goal": gl}, "actions": acts[torch.from_numpy(s)].clone(),
                "next_observations": {"observation": nxt, "goal": gl}, "rewards": torch.from_numpy(out64[0].copy()),
                "terminals": torch.from_numpy(out64[1].copy())}
    states = {}
    for m in modalities:
        win = np.stack([TO.pad_frames(torch.from_numpy(frames[m][s[b]:s[b] + w[b]]), int(w[b]), T).numpy()
                        for b in range(B)])
        states[m] = torch.from_numpy(shifted(m, win, 0).copy())
    pad_fn = TO.pad_rel_actions if zero_pad else TO.pad_frames
    act = torch.stack([pad_fn(acts[s[b]:s[b] + w[b]], int(w[b]), T) for b in range(B)])
    batch = {"states": states, "actions": act, "idx": torch.from_numpy(out64[0].copy()),
             "window_size": torch.from_numpy(out64[1].copy())}
    if kind == TACORL:
        batch["goal"] = {m: single(m, goal, T) for m in modalities}
        batch["disp"] = torch.from_numpy(out64[2].copy())
    return batch
