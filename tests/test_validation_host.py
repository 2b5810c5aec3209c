"""Host tests of validation sweeps (DESIGN.md section 14): the items a sweep visits, its batch / tail layout, the
refusals of a sweep-mode replay, and the item-weighted aggregation of the logged scalars."""
import numpy as np
import pytest
import torch

from tests import sweep_oracle as SO

LENGTHS = [12, 5, 30, 1, 9, 3, 20, 2, 17]


def _episodes(lengths=LENGTHS, seed=0):
    g = np.random.default_rng(seed)
    eps = []
    for n in lengths:
        eps.append({"rgb_static": g.integers(0, 256, (n, 4, 4, 3), dtype=np.uint8),
                    "rel_actions": g.uniform(-1, 1, (n, 7)).astype(np.float32)})
    return eps


def _global_items(index, kind, min_window):
    """(episode id, offset in the episode) of every item of the rank, in store order."""
    starts = np.concatenate([[0], np.cumsum(index.episode_lengths)[:-1]])
    out = []
    for f in index.items(kind, min_window):
        e = int(np.searchsorted(starts, f, side="right")) - 1
        out.append((index.episode_ids[e], int(f - starts[e])))
    return out


@pytest.mark.parametrize("kind", ["play_lmp", "tacorl", "cql"])
def test_a_sweep_visits_every_item_of_the_rank_once_and_the_ranks_cover_the_split(kind):
    from tacorl_b200.replay import ReplayIndex
    eps = _episodes()
    whole = ReplayIndex(eps)
    union = []
    for rank in range(3):
        ix = ReplayIndex(eps, rank=rank, world_size=3)
        batches = SO.sweep(kind, ix, 4, seed=7, min_window=3, max_window=6)
        starts = np.concatenate([b["tab"][0] for b in batches])
        assert starts.tolist() == ix.items(kind, 3).tolist()          # each item once, in store order
        again = SO.sweep(kind, ix, 4, seed=7, min_window=3, max_window=6)
        for a, b in zip(batches, again):
            assert np.array_equal(a["tab"], b["tab"]) and np.array_equal(a["out64"], b["out64"])
        union += _global_items(ix, kind, 3)
    assert len(union) == len(set(union))
    assert sorted(union) == sorted(_global_items(whole, kind, 3))


def test_sweep_draws_follow_the_training_laws():
    """Windows within [min_window, min(max_window, frames left)], goals inside the episode or negative."""
    from tacorl_b200.replay import ReplayIndex
    ix = ReplayIndex(_episodes())
    for t in SO.sweep("tacorl", ix, 8, seed=3, min_window=2, max_window=6, neg_frac=0.3):
        s, w, goal, disp = (t["tab"][i].astype(np.int64) for i in range(4))
        end = ix.ep_end[s]
        assert ((w >= 2) & (w <= np.minimum(6, end - s + 1))).all()
        pos = disp >= 1
        assert ((goal[pos] >= s[pos] + w[pos] - 1) & (goal[pos] <= end[pos])).all()
        assert (disp[~pos] == -1).all()
    for t in SO.sweep("cql", ix, 8, seed=3, goal_p=0.5):
        s, goal, hit = t["tab"][0].astype(np.int64), t["tab"][2].astype(np.int64), t["tab"][3]
        assert ((goal > s) & (goal <= ix.ep_end[s])).all() and (hit == (goal == s + 1)).all()


def test_sweep_draws_differ_from_item_to_item_and_not_with_the_batch_size():
    from tacorl_b200.replay import ReplayIndex
    ix = ReplayIndex(_episodes())
    a = np.concatenate([t["tab"] for t in SO.sweep("play_lmp", ix, 4, seed=1, min_window=1, max_window=8)], 1)
    b = np.concatenate([t["tab"] for t in SO.sweep("play_lmp", ix, 7, seed=1, min_window=1, max_window=8)], 1)
    assert np.array_equal(a, b)
    assert len(set(a[1].tolist())) > 1


def test_tail_sizes():
    from tacorl_b200.replay import ReplayIndex, sweep_shape
    assert sweep_shape(5, 8) == (0, 5)                   # items < B: the tail is the whole sweep
    assert sweep_shape(24, 8) == (3, 0)                  # items % B == 0: no tail
    assert sweep_shape(25, 8) == (3, 1)
    # an episode shorter than min_window contributes no window start; CQL counts transitions
    ix = ReplayIndex(_episodes([6, 2, 5]))
    assert len(ix.items("play_lmp", 3)) == 4 + 0 + 3
    assert len(ix.items("cql")) == 5 + 1 + 4
    assert sweep_shape(len(ix.items("play_lmp", 3)), 4) == (1, 3)
    batches = SO.sweep("play_lmp", ix, 4, seed=0, min_window=3, max_window=4)
    assert [b["tab"].shape[1] for b in batches] == [4, 3]


def test_sweep_mode_refuses_augmentation_and_use_as_a_training_source():
    from tacorl_b200 import trainer as TR
    from tacorl_b200.replay import DeviceReplay, ReplayIndex
    ix = ReplayIndex(_episodes())
    with pytest.raises(ValueError, match="does not augment"):
        DeviceReplay(ix, 4, mode="sweep", pad=2)
    with pytest.raises(ValueError, match="does not augment"):
        DeviceReplay(ix, 4, mode="sweep", jitter={"brightness": 0.1})
    with pytest.raises(ValueError, match="mode"):
        DeviceReplay(ix, 4, mode="eval")
    sweep = DeviceReplay.__new__(DeviceReplay)           # no device needed: refused before anything is set up
    sweep.mode = "sweep"
    with pytest.raises(ValueError, match="pass it as val="):
        TR.Trainer(max_steps=1, device=torch.device("cuda", 0)).fit(torch.nn.Linear(1, 1), sweep)
    train = DeviceReplay.__new__(DeviceReplay)
    train.mode = "train"
    with pytest.raises(ValueError, match="mode='sweep'"):
        TR.Trainer(max_steps=1, device=torch.device("cuda", 0))._check_val(train)
    with pytest.raises(ValueError, match="check_val_every_n_epoch"):
        TR.Trainer(check_val_every_n_epoch=0)


def test_item_weighted_means_match_a_hand_computation():
    from tacorl_b200.runtime import item_weighted_means
    keys = ["validation/a", "validation/b"]
    # rank 0: batches of 4 and 1 items; rank 1: one batch of 3
    r0 = [(4, [1.0, 10.0]), (1, [6.0, -2.0])]
    r1 = [(3, [4.0, 0.5])]

    def vec(batches):
        sums = [sum(n * v[i] for n, v in batches) for i in range(len(keys))]
        return sums + [sum(n for n, _ in batches)]
    got = item_weighted_means(keys, [vec(r0), vec(r1)])
    assert got["validation/a"] == pytest.approx((4 * 1.0 + 1 * 6.0 + 3 * 4.0) / 8)
    assert got["validation/b"] == pytest.approx((4 * 10.0 - 2.0 + 1.5) / 8)
    # not the mean of the batch means, nor of the rank means
    assert got["validation/a"] != pytest.approx((1.0 + 6.0 + 4.0) / 3)
    assert got["validation/a"] != pytest.approx(((4 + 6) / 5 + 4.0) / 2)
    with pytest.raises(ValueError):
        item_weighted_means(keys, [[1.0, 2.0, 0.0]])
    with pytest.raises(ValueError):
        item_weighted_means(keys, [[1.0, 2.0]])
