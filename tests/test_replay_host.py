"""Host-side tests of the HBM-resident replay: ReplayIndex loading and sharding, the numpy restatement of the device
sampler (oracle/replay_oracle.py) and its statistics, and the memory check of DeviceReplay.  No GPU needed."""
import numpy as np
import pytest
import torch
from scipy import stats

from oracle import replay_oracle as RO
from oracle import transforms_oracle as TO

EPISODES = [(0, 9), (10, 12), (13, 30), (31, 31), (32, 47)]      # inclusive [start, end] frame ids


def _frame(i, h, w):
    g = np.random.default_rng(i + 1000)
    return g.integers(0, 256, (h, w, 3), dtype=np.uint8)


@pytest.fixture
def calvin_dir(tmp_path):
    """A tiny CALVIN-format split: ep_start_end_ids.npy + one episode_{id:07d}.npz per frame (ids start at 100 so that
    frame ids and store positions differ)."""
    off = 100
    np.save(tmp_path / "ep_start_end_ids.npy", np.array([[s + off, e + off] for s, e in EPISODES[::-1]]))
    for s, e in EPISODES:
        for i in range(s + off, e + off + 1):
            np.savez(tmp_path / f"episode_{i:07d}.npz", rgb_static=_frame(i, 12, 16), rgb_gripper=_frame(-i, 8, 8),
                     rel_actions=np.full(7, i, np.float64), actions=np.full(7, -i, np.float64))
    return tmp_path, off


def test_philox_matches_the_random123_known_answers():
    assert [int(v) for v in RO.philox4x32_10(0, 0, 0, 0, 0, 0)] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    ff = 0xFFFFFFFF
    assert [int(v) for v in RO.philox4x32_10(ff, ff, ff, ff, ff, ff)] == [0x408F276D, 0x41C83B0E, 0xA20BC7C6,
                                                                          0x6D5451FD]
    got = RO.philox4x32_10(0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344, 0xA4093822, 0x299F31D0)
    assert [int(v) for v in got] == [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


def test_calvin_directory_loads_exactly(calvin_dir):
    from tacorl_b200.replay import ReplayIndex
    root, off = calvin_dir
    ix = ReplayIndex.from_calvin(root, modalities=("rgb_static", "rgb_gripper"))
    ids = np.arange(48) + off
    assert ix.num_frames == 48 and ix.episode_ids == [s + off for s, _ in EPISODES]
    assert ix.frames["rgb_static"].shape == (48, 3, 12, 16) and ix.frames["rgb_gripper"].shape == (48, 3, 8, 8)
    for f in (0, 11, 31, 47):
        assert np.array_equal(ix.frames["rgb_static"][f], _frame(ids[f], 12, 16).transpose(2, 0, 1))
        assert np.array_equal(ix.frames["rgb_gripper"][f], _frame(-ids[f], 8, 8).transpose(2, 0, 1))
    assert np.array_equal(ix.actions[:, 0], ids.astype(np.float32)) and ix.actions.dtype == np.float32
    want_end = np.concatenate([np.full(e - s + 1, e) for s, e in EPISODES])
    assert np.array_equal(ix.ep_end, want_end)
    assert np.array_equal(ix.valid_starts(4), [f for f in range(48) if want_end[f] - f + 1 >= 4])
    assert np.array_equal(ix.valid_transitions(), [f for f in range(48) if want_end[f] > f])
    assert ix.nbytes == 48 * (3 * 12 * 16 + 3 * 8 * 8 + 7 * 4 + 4)
    absolute = ReplayIndex.from_calvin(root, action_key="actions")
    assert np.array_equal(absolute.actions[:, 0], -ids.astype(np.float32))
    small = ReplayIndex.from_calvin(root, resize={"rgb_static": (6, 8)})
    assert small.frames["rgb_static"].shape == (48, 3, 6, 8)


def test_rank_shards_are_disjoint_cover_every_episode_and_balance(calvin_dir):
    from tacorl_b200.replay import ReplayIndex, shard_episodes
    root, off = calvin_dir
    lengths = [e - s + 1 for s, e in EPISODES]
    for world in (1, 2, 3, 5):
        shards = shard_episodes(lengths, world)
        flat = sorted(e for s in shards for e in s)
        assert flat == list(range(len(EPISODES)))
        loads = [sum(lengths[e] for e in s) for s in shards]
        assert max(loads) - min(loads) <= max(lengths)
    g = np.random.default_rng(0)
    big = list(g.integers(1, 500, 301))
    loads = [sum(big[e] for e in s) for s in shard_episodes(big, 8)]
    assert max(loads) - min(loads) <= max(big)
    with pytest.raises(ValueError):
        shard_episodes(lengths, 6)
    parts = [ReplayIndex.from_calvin(root, rank=r, world_size=2) for r in range(2)]
    assert sorted(parts[0].episode_ids + parts[1].episode_ids) == [s + off for s, _ in EPISODES]
    assert not set(parts[0].episode_ids) & set(parts[1].episode_ids)
    assert sum(p.num_frames for p in parts) == 48
    for p in parts:      # per-rank stores are self-contained: ep_end stays inside the rank's frames
        assert (p.ep_end < p.num_frames).all()


def test_index_from_arrays_matches_the_calvin_loader(calvin_dir):
    from tacorl_b200.replay import ReplayIndex
    root, off = calvin_dir
    eps = [{"rgb_static": np.stack([_frame(i + off, 12, 16) for i in range(s, e + 1)]),
            "rel_actions": np.stack([np.full(7, i + off, np.float32) for i in range(s, e + 1)])} for s, e in EPISODES]
    a = ReplayIndex(eps)
    b = ReplayIndex.from_calvin(root)
    assert np.array_equal(a.frames["rgb_static"], b.frames["rgb_static"])
    assert np.array_equal(a.actions, b.actions) and np.array_equal(a.ep_end, b.ep_end)


def _index(lengths, seed=0):
    ends = np.cumsum(lengths) - 1
    return np.repeat(ends, lengths).astype(np.int64)


def test_oracle_draws_stay_in_episode_and_follow_their_laws():
    """10^5 draws at a fixed seed: no window crosses an episode end, starts are uniform over the valid starts (chi^2),
    window sizes are uniform on their range, and the goal offsets follow Geometric(goal_p)."""
    lengths = [40, 7, 25, 3, 60, 16, 9]
    ep_end = _index(lengths)
    F = len(ep_end)
    minw, maxw, p = 4, 16, 0.3
    valid = np.nonzero(ep_end - np.arange(F) + 1 >= minw)[0]
    thr = RO.geometric_thresholds(p)
    starts, dists, sizes_at_full, negs = [], [], [], []
    for step in range(100):
        t = RO.sample("tacorl", step, 1000, 7, 0, ep_end, valid, min_window=minw, max_window=maxw, geom_thr=thr,
                      neg_thr=int(0.1 * 2 ** 32))
        s, w, goal, disp = (t["tab"][i].astype(np.int64) for i in range(4))
        assert (w >= minw).all() and (w <= maxw).all()
        assert (s + w - 1 <= ep_end[s]).all()                             # the window stays inside its episode
        pos = disp > 0
        assert (goal[pos] <= ep_end[s[pos]]).all() and (goal[pos] >= s[pos] + w[pos] - 1).all()
        assert np.array_equal(disp[pos], goal[pos] - (s[pos] + w[pos] - 1) + 1)
        assert ((goal >= 0) & (goal < F)).all()
        starts.append(s)
        negs.append(disp == -1)
        # unclipped goal offsets: where the episode has more room than any draw we observe
        room = ep_end[s] - (s + w - 1)
        dists.append(disp[pos & (disp <= room)])
        full = ep_end[s] - s + 1 >= maxw
        sizes_at_full.append(w[full])
    starts = np.concatenate(starts)
    counts = np.bincount(np.searchsorted(valid, starts), minlength=len(valid))
    assert np.array_equal(np.unique(starts), valid)
    assert stats.chisquare(counts).pvalue > 1e-3
    sizes = np.concatenate(sizes_at_full)
    assert stats.chisquare(np.bincount(sizes - minw, minlength=maxw - minw + 1)).pvalue > 1e-3
    assert abs(np.concatenate(negs).mean() - 0.1) < 0.005
    d = np.concatenate(dists)
    # geometric draws before clipping: compare the raw law on the same uniforms instead
    u = np.concatenate([RO.philox4x32_10(s_, 0, np.arange(1000), 0, *RO.key(7, 0))[3] for s_ in range(100)])
    raw = RO.geometric(u, thr)
    kk = np.arange(1, 12)
    want = p * (1 - p) ** (kk - 1)
    obs = np.array([(raw == k).sum() for k in kk] + [(raw >= 12).sum()])
    exp = np.append(want, 1 - want.sum()) * len(raw)
    assert stats.chisquare(obs, exp).pvalue > 1e-3
    assert d.min() >= 1
    # CQL: k ~ Geometric(goal_p), goal = min(i + k, ep_end[i]); reward = terminal = [goal == i + 1]
    tv = np.nonzero(ep_end > np.arange(F))[0]
    t = RO.sample("cql", 3, 100000, 11, 1, ep_end, tv, geom_thr=thr)
    i, goal, hit = t["tab"][0].astype(np.int64), t["tab"][2].astype(np.int64), t["tab"][3]
    assert np.isin(i, tv).all() and (i + 1 <= ep_end[i]).all()
    assert (goal <= ep_end[i]).all() and (goal > i).all()
    assert np.array_equal(hit, (goal == i + 1).astype(np.int32))
    assert np.array_equal(t["out64"][0], t["out64"][1])
    room = ep_end[i] - i
    k = (goal - i)[room >= 12]
    obs = np.array([(k == j).sum() for j in kk])
    assert stats.chisquare(np.append(obs, (k >= 12).sum()), np.append(want, 1 - want.sum()) * len(k)).pvalue > 1e-3
    assert abs(hit[room >= 2].mean() - p) < 0.01          # (a transition ending its episode always hits)


def test_oracle_is_deterministic_and_separates_seeds_ranks_and_steps():
    ep_end = _index([30, 30])
    valid = np.arange(50)
    kw = dict(min_window=4, max_window=8, n_mod=2, n_slots=8, pad=3)
    a = RO.sample("play_lmp", 5, 64, 1, 0, ep_end, valid, **kw)
    assert np.array_equal(a["tab"], RO.sample("play_lmp", 5, 64, 1, 0, ep_end, valid, **kw)["tab"])
    for other in (RO.sample("play_lmp", 6, 64, 1, 0, ep_end, valid, **kw),
                  RO.sample("play_lmp", 5, 64, 2, 0, ep_end, valid, **kw),
                  RO.sample("play_lmp", 5, 64, 1, 1, ep_end, valid, **kw)):
        assert not np.array_equal(a["tab"], other["tab"]) and not np.array_equal(a["shift"], other["shift"])
    assert a["shift"].shape == (2, 64, 8, 2) and a["shift"].min() >= 0 and a["shift"].max() <= 6


def test_integer_shift_is_random_shifts_aug():
    g = torch.Generator().manual_seed(0)
    x = torch.randint(0, 256, (5, 3, 20, 20), generator=g, dtype=torch.uint8)
    pad = 4
    sh = torch.randint(0, 2 * pad + 1, (5, 2), generator=g)
    want = TO.random_shifts(x.float(), pad, sh.view(5, 1, 1, 2)).round().to(torch.uint8)
    assert np.array_equal(RO.shift_frames(x.numpy(), sh.numpy(), pad), want.numpy())


def test_product_geometric_table_equals_the_oracle_one():
    from tacorl_b200.replay import geometric_thresholds
    for p in (0.05, 0.3, 0.9, 1.0):
        a, b = geometric_thresholds(p), RO.geometric_thresholds(p)
        assert a.dtype == np.uint32 and np.array_equal(a, b)
        assert (np.diff(a.astype(np.int64)) >= 0).all() and int(a[-1]) == 2 ** 32 - 1


def test_memory_check_raises_before_any_allocation(monkeypatch):
    from tacorl_b200.replay import DeviceReplay, ReplayIndex
    eps = [{"rgb_static": np.zeros((20, 8, 8, 3), np.uint8), "rel_actions": np.zeros((20, 7), np.float32)}]
    ix = ReplayIndex(eps)
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (1000, 2000))

    def no_alloc(*a, **k):
        raise AssertionError("allocated before the memory check")
    monkeypatch.setattr(torch, "empty", no_alloc)
    monkeypatch.setattr(torch, "zeros", no_alloc)
    with pytest.raises(MemoryError, match=r"needs \d+ bytes .* only 1000 of 2000"):
        DeviceReplay(ix, 4, kind="play_lmp", min_window=2, max_window=4, device="cuda:0")


def test_geometric_table_refuses_to_cut_the_law_off():
    from tacorl_b200.replay import geometric_thresholds
    with pytest.raises(ValueError, match="beyond d = 4096"):
        geometric_thresholds(0.001)
    assert int(geometric_thresholds(0.01)[-1]) == 2 ** 32 - 1


def test_negative_goal_fraction_one_is_every_draw():
    ep_end = _index([30, 30])
    t = RO.sample("tacorl", 0, 4096, 3, 0, ep_end, np.arange(50), min_window=4, max_window=8,
                  geom_thr=RO.geometric_thresholds(0.3), neg_thr=2 ** 32)
    assert (t["tab"][3] == -1).all()


def test_jitter_factor_draws_are_float32_exact_and_in_range():
    u = np.array([0, 255, 256, 2 ** 31, 2 ** 32 - 1], dtype=np.uint32)
    f = RO.uniform_float(u, np.float32(0.9), np.float32(0.2))
    assert f.dtype == np.float32 and f[0] == np.float32(0.9) and f[1] == np.float32(0.9) and (f < 1.1).all()
    ep_end = _index([30, 30])
    jit = {"ops": 0b1011, "lo": [0.9, 0.9, -0.02], "span": [0.2, 0.2, 0.04]}
    t = RO.sample("play_lmp", 1, 64, 3, 0, ep_end, np.arange(50), min_window=4, max_window=8, n_mod=2, n_slots=8,
                  pad=0, jitter=jit)
    orders = {tuple(RO.unpack_order(c)) for c in t["jit_order"].reshape(-1)}
    assert orders == {(0, 1, 3), (0, 3, 1), (1, 0, 3), (1, 3, 0), (3, 0, 1), (3, 1, 0)}
    fac = t["jit_factors"]
    assert fac.shape == (2, 64, 8, 3) and (fac[..., :2] >= 0.9).all() and (fac[..., 2] >= -0.02).all()
    only_hue = RO.sample("play_lmp", 1, 64, 3, 0, ep_end, np.arange(50), min_window=4, max_window=8, n_mod=1,
                         n_slots=8, jitter={"ops": 8, "lo": [0, 0, -0.02], "span": [0, 0, 0.04]})
    assert {tuple(RO.unpack_order(c)) for c in only_hue["jit_order"].reshape(-1)} == {(3,)}
    assert (only_hue["jit_factors"][..., :2] == 1).all()


def test_replay_device_defaults_to_the_local_rank(monkeypatch):
    from tacorl_b200.replay import DeviceReplay, ReplayIndex
    eps = [{"rgb_static": np.zeros((20, 8, 8, 3), np.uint8), "rel_actions": np.zeros((20, 7), np.float32)}]
    seen = []
    monkeypatch.setenv("LOCAL_RANK", "3")
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (seen.append(device), (0, 1))[1])
    with pytest.raises(MemoryError, match="on cuda:3"):
        DeviceReplay(ReplayIndex(eps), 4, min_window=2, max_window=4)
    assert seen == [torch.device("cuda", 3)]
