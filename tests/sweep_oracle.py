"""TEST INFRASTRUCTURE — numpy restatement of a validation sweep (DESIGN.md section 14): the items a sweep visits and
the tables replay_sample_kernel writes in sweep mode.  The draws are those of oracle/replay_oracle.py with the counter
(lo32(item), hi32(item), 0, draw id) in place of (lo32(step), hi32(step), sample, draw id); the assembly is
replay_oracle.assemble over the n rows."""
import numpy as np

from oracle import replay_oracle as RO


def sweep_tables(kind, cursor, n, seed, rank, ep_end, valid, *, min_window=1, max_window=1, geom_thr=None, neg_thr=0):
    """Rows [0, n) of the tables of one sweep batch starting at item `cursor`: int32 `tab` (4, n), int64 `out64`
    (3, n)."""
    kind = RO.KINDS.get(kind, kind)
    k0, k1 = RO.key(seed, rank)
    valid = np.asarray(valid, dtype=np.int64)
    item = (int(cursor) + np.arange(n, dtype=np.uint64)) % np.uint64(len(valid))
    lo, hi = item & np.uint64(0xFFFFFFFF), item >> np.uint64(32)
    r = RO.philox4x32_10(lo, hi, 0, RO.DRAW_SAMPLE, k0, k1)
    ep_end = np.asarray(ep_end, dtype=np.int64)
    s = valid[item.astype(np.int64)]
    end = ep_end[s]
    if kind == RO.CQL:
        goal = np.minimum(s + RO.geometric(r[3], geom_thr), end)
        hit = (goal == s + 1).astype(np.int64)
        return {"tab": np.stack([s, np.ones(n, np.int64), goal, hit]).astype(np.int32),
                "out64": np.stack([hit, hit, goal]).astype(np.int64), "shift": None}
    wmax = np.minimum(max_window, end - s + 1)
    w = min_window + ((r[1].astype(np.uint64) * (wmax - min_window + 1).astype(np.uint64)) >> np.uint64(32)).astype(np.int64)
    last = s + w - 1
    goal, disp = last.copy(), np.ones(n, np.int64)
    if kind == RO.TACORL:
        neg = r[2].astype(np.int64) < int(neg_thr)
        g = RO.philox4x32_10(lo, hi, 0, RO.DRAW_NEG_GOAL, k0, k1)
        pos_goal = np.minimum(last + RO.geometric(r[3], geom_thr) - 1, end)
        goal = np.where(neg, RO.uniform_below(g[0], len(ep_end)), pos_goal)
        disp = np.where(neg, -1, goal - last + 1)
    return {"tab": np.stack([s, w, goal, disp]).astype(np.int32), "out64": np.stack([s, w, disp]).astype(np.int64),
            "shift": None}


def sweep(kind, index, B, seed, *, min_window=1, max_window=1, goal_p=0.3, neg_frac=0.1):
    """Every batch of one sweep of a ReplayIndex: a list of table dicts, `items // B` full ones then the tail."""
    valid = index.items(kind, min_window)
    geom = RO.geometric_thresholds(goal_p)
    neg_thr = int(np.floor(neg_frac * 2.0 ** 32)) if kind == "tacorl" else 0
    out, cursor = [], 0
    while cursor < len(valid):
        n = min(B, len(valid) - cursor)
        out.append(sweep_tables(kind, cursor, n, seed, index.rank, index.ep_end, valid, min_window=min_window,
                                max_window=max_window, geom_thr=geom, neg_thr=neg_thr))
        cursor += n
    return out
