"""GPU tests of the HBM-resident replay (tacorl_b200/replay.py, csrc/replay.cu) against its numpy restatement
(oracle/replay_oracle.py), and of the training paths it feeds: eager steps, CUDA-graph replays and Trainer.fit."""
import numpy as np
import pytest
import torch

from oracle import replay_oracle as RO
from oracle import synth as S
from oracle import tacorl_oracle as O
from tests.gpu_util import DEV, build_cql_flat, build_play_lmp, build_tacorl, cql_tape, play_lmp_tape, tacorl_tape, to_dev

pytestmark = pytest.mark.gpu

# short episodes (shorter than the longest window), a single-frame one, and long ones: windows shorter than T, goals
# clipped to the episode end and transitions next to episode ends all occur at these batch sizes
LENGTHS = [12, 5, 30, 1, 9, 3, 20, 2, 17]


def _episodes(shapes, seed=0, lengths=LENGTHS):
    g = np.random.default_rng(seed)
    eps = []
    for n in lengths:
        ep = {m: g.integers(0, 256, (n, h, w, 3), dtype=np.uint8) for m, (h, w) in shapes.items()}
        act = g.uniform(-1, 1, (n, 7)).astype(np.float32)
        act[:, -1] = np.where(act[:, -1] > 0, 1.0, -1.0)
        ep["rel_actions"] = act
        eps.append(ep)
    return eps


@pytest.fixture(scope="module")
def two_view_index():
    from tacorl_b200.replay import ReplayIndex
    return ReplayIndex(_episodes({"rgb_static": (24, 36), "rgb_gripper": (12, 12)}),
                       modalities=("rgb_static", "rgb_gripper"))


def _replay(index, kind, **kw):
    from tacorl_b200.replay import DeviceReplay
    args = dict(batch_size=16, kind=kind, min_window=2, max_window=8, pad=3, goal_p=0.3, neg_frac=0.25, seed=11,
                device=DEV)
    args.update(kw)
    return DeviceReplay(index, **args)


JITTER = {"brightness": 0.1, "contrast": 0.1, "hue": 0.02}


def _oracle_tables(r, step):
    ix = r.index
    valid = ix.valid_transitions() if r.kind == "cql" else ix.valid_starts(r.min_window)
    return RO.sample(r.kind, step, r.B, r.seed, r.rank, ix.ep_end, valid, min_window=r.min_window,
                     max_window=r.max_window, geom_thr=RO.geometric_thresholds(r.goal_p), neg_thr=r.neg_thr,
                     n_mod=len(ix.modalities), n_slots=r.n_slots, pad=r.pad, jitter=r.jitter)


def _cpu(batch):
    return {k: _cpu(v) if isinstance(v, dict) else v.detach().cpu().clone() for k, v in batch.items()}


def _assert_batches_equal(got, want, path=""):
    assert set(got) == set(want), (path, set(got) ^ set(want))
    for k in want:
        if isinstance(want[k], dict):
            _assert_batches_equal(got[k], want[k], path + "." + k)
        else:
            g, w = got[k], want[k]
            assert g.dtype == w.dtype and g.shape == w.shape, (path + "." + k, g.dtype, w.dtype, g.shape, w.shape)
            assert torch.equal(g, w), (path + "." + k, int((g != w).sum()))


@pytest.mark.parametrize("kind", ["play_lmp", "tacorl", "cql"])
@pytest.mark.parametrize("seed", [0, 11, 2 ** 40 + 3])
def test_sampler_tables_equal_the_oracle_bit_for_bit(two_view_index, kind, seed):
    r = _replay(two_view_index, kind, seed=seed, jitter=JITTER if seed != 0 else {"hue": 0.05})
    for step in list(range(4)) + [2 ** 32 + 5]:
        if step > 3:
            r.load_state_dict({"step": step})
        r.sample()
        want = _oracle_tables(r, step)
        assert np.array_equal(r.tab.cpu().numpy(), want["tab"]), (kind, seed, step)
        assert np.array_equal(r.out64.cpu().numpy(), want["out64"]), (kind, seed, step)
        assert np.array_equal(r.shift.cpu().numpy(), want["shift"]), (kind, seed, step)
        assert np.array_equal(r.jit_order.cpu().numpy(), want["jit_order"]), (kind, seed, step)
        assert np.array_equal(r.jit_factors.cpu().numpy().view(np.int32), want["jit_factors"].view(np.int32))
        assert r.step == step + 1


def test_negative_goal_fraction_one_makes_every_goal_negative(two_view_index):
    r = _replay(two_view_index, "tacorl", neg_frac=1.0, batch_size=64)
    for step in range(3):
        r.sample()
        assert (r.out64[2] == -1).all()
        assert np.array_equal(r.tab.cpu().numpy(), _oracle_tables(r, step)["tab"])


@pytest.mark.parametrize("kind", ["play_lmp", "tacorl", "cql"])
def test_jittered_batch_matches_torchvision_ops_on_the_assembled_frames(two_view_index, kind):
    """jitter on: float32 frames = ScaleImageTensor -> ColorJitter(drawn order, factors) -> Normalize of the uint8
    frames the gather assembles, within test_color_jitter_matches_torchvision_ops's tolerance."""
    r = _replay(two_view_index, kind, jitter=dict(JITTER, mean=0.5, std=0.5), batch_size=6)
    ix = r.index
    for step in range(2):
        got = _cpu(r.sample())
        t = _oracle_tables(r, step)
        want_u8 = RO.assemble(kind, t, ix.frames, ix.actions, r.T, r.pad, list(ix.modalities))
        mods = list(ix.modalities)

        def check(g, w, m, slot0):
            mi = mods.index(m)
            nf = w.shape[1] if w.dim() == 5 else 1
            w = w.reshape(-1, *w.shape[-3:])
            order = t["jit_order"][mi][:, slot0:slot0 + nf].reshape(-1)
            fac = t["jit_factors"][mi][:, slot0:slot0 + nf].reshape(-1, 3)
            ref = RO.jitter_frames(w.numpy(), order, fac)
            assert g.dtype == torch.float32
            err = float((g.reshape(ref.shape) - ref).abs().max())
            assert err < 1e-4, (kind, m, err)

        for m in mods:
            if kind == "cql":
                check(got["observations"]["observation"][m], want_u8["observations"]["observation"][m], m, 0)
                check(got["next_observations"]["observation"][m], want_u8["next_observations"]["observation"][m], m, 1)
                check(got["observations"]["goal"][m], want_u8["observations"]["goal"][m], m, 2)
            else:
                check(got["states"][m], want_u8["states"][m], m, 0)
                if kind == "tacorl":
                    check(got["goal"][m], want_u8["goal"][m], m, r.T)
        assert torch.equal(got["actions"], want_u8["actions"])


@pytest.mark.parametrize("kind", ["play_lmp", "tacorl", "cql"])
@pytest.mark.parametrize("pad", [0, 3])
def test_assembled_batch_equals_the_oracle_assembly(two_view_index, kind, pad):
    """Two modalities at different resolutions (24x36 and 12x12), short windows, clipped goals: byte for byte."""
    r = _replay(two_view_index, kind, pad=pad, batch_size=24)
    ix = r.index
    saw_short = saw_clipped = False
    for step in range(3):
        got = _cpu(r.sample())
        tables = {"tab": r.tab.cpu().numpy(), "out64": r.out64.cpu().numpy(),
                  "shift": None if r.shift is None else r.shift.cpu().numpy()}
        want = RO.assemble(kind, tables, ix.frames, ix.actions, r.T, pad, list(ix.modalities))
        _assert_batches_equal(got, want)
        s, w, goal = tables["tab"][0], tables["tab"][1], tables["tab"][2]
        saw_short |= bool((w < r.max_window).any())
        saw_clipped |= bool((goal == ix.ep_end[s]).any())
    assert saw_clipped and (kind == "cql" or saw_short)


def test_eager_step_k_equals_graph_replay_k(two_view_index):
    from tacorl_b200 import runtime
    r = _replay(two_view_index, "tacorl")
    eager = [_cpu(r.sample()) for _ in range(4)]
    r.load_state_dict({"step": 0})
    seen = []
    g = runtime.GraphedTrainStep(lambda b: None, None, device=torch.device(DEV), warmup=2, source=r)
    assert r.step == 0                                   # capture warm-up consumed no draws
    for k in range(4):
        g()
        seen.append(_cpu(r.batch()))
        _assert_batches_equal(seen[k], eager[k])
    assert r.step == 4
    with pytest.raises(ValueError):
        g(eager[0])


def _play_module(T):
    m = build_play_lmp("tanh_net", ("rgb_static",), 64, 16, T)
    shapes = {k: list(v.shape) for k, v in m.state_dict().items()}
    m.load_state_dict(S.synth_state_dict(shapes, 4))
    m.to(DEV)
    return m


def _tacorl_module(T):
    lmp = build_play_lmp("tanh_net", ("rgb_static",), 64, 16, T)
    t = build_tacorl(lmp)
    shapes = {k: list(v.shape) for k, v in t.state_dict().items()}
    t.load_state_dict(S.synth_state_dict(shapes, 6))
    t.to(DEV)
    t.optimizers()
    return t


def _cql_module():
    m = build_cql_flat()
    shapes = {k: list(v.shape) for k, v in m.state_dict().items()}
    m.load_state_dict(S.synth_state_dict(shapes, 29))
    m.to(DEV)
    m.train()
    m.optimizers()
    return m


@pytest.mark.parametrize("kind", ["play_lmp", "tacorl", "cql"])
def test_replay_fed_step_equals_host_fed_step_bit_for_bit(kind):
    """fp32: the same step fed by DeviceReplay and fed the same batch as a host dict gives the same loss and parameters,
    bit for bit, under the same noise tape."""
    from tacorl_b200 import ops
    from tacorl_b200.replay import ReplayIndex
    from tacorl_b200.utils.rng import noise_tape
    ops.set_precision("fp32")
    T, B = 8, 3
    ix = ReplayIndex(_episodes({"rgb_static": (84, 84)}, seed=5))
    r = _replay(ix, kind, batch_size=B, min_window=4, max_window=T, pad=4, seed=3)
    torch.manual_seed(1)
    if kind == "play_lmp":
        noise = O.draw_play_lmp_noise(B, T)
        tape = lambda: play_lmp_tape(noise, B)
    elif kind == "tacorl":
        noise = O.draw_tacorl_noise(B)
        tape = lambda: tacorl_tape(noise)
    else:
        noise = O.draw_cql_noise(B)
        tape = lambda: cql_tape(noise)

    def run(batch):
        m = {"play_lmp": lambda: _play_module(T), "tacorl": lambda: _tacorl_module(T), "cql": _cql_module}[kind]()
        with noise_tape(tape()):
            if kind == "play_lmp":
                opt = m.configure_optimizers()
                loss = m.training_step(batch, 0)
                loss.backward()
                opt.step()
            else:
                m.training_step(batch)
                loss = m.logged["train/q1_loss"]
        torch.cuda.synchronize()
        return float(loss.detach()), {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}

    dev_batch = r.sample()
    host = _cpu(dev_batch)
    l_dev, sd_dev = run(dev_batch)
    l_host, sd_host = run(to_dev(host))
    assert l_dev == l_host
    assert [k for k in sd_dev if not torch.equal(sd_dev[k], sd_host[k])] == []


def test_graph_launches_grow_by_the_two_replay_kernels_and_no_h2d_copy():
    from torch.profiler import ProfilerActivity, profile

    from tacorl_b200 import ops, runtime
    from tacorl_b200.replay import ReplayIndex
    ops.set_precision("fp32")
    T = 8
    ix = ReplayIndex(_episodes({"rgb_static": (84, 84)}, seed=6))
    r = _replay(ix, "play_lmp", batch_size=2, min_window=4, max_window=T, pad=4)
    m = _play_module(T)
    opt = m.configure_optimizers()
    fed = runtime.GraphedTrainStep(runtime.play_lmp_step_fn(m, opt), _cpu(r.batch()), warmup=2)
    own = runtime.GraphedTrainStep(runtime.play_lmp_step_fn(m, opt), None, warmup=2, source=r)
    assert own.launches_per_replay == fed.launches_per_replay + 2 == fed.launches_per_replay + r.launches_per_sample
    rj = _replay(ix, "play_lmp", batch_size=2, min_window=4, max_window=T, pad=4, jitter=JITTER)
    fed_f = runtime.GraphedTrainStep(runtime.play_lmp_step_fn(m, opt), _cpu(rj.batch()), warmup=2)
    own_j = runtime.GraphedTrainStep(runtime.play_lmp_step_fn(m, opt), None, warmup=2, source=rj)
    assert own_j.launches_per_replay == fed_f.launches_per_replay + 4
    own()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            own()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert names
    assert not [n for n in names if "HtoD" in n or "Host to Device" in n], sorted(set(names))[:40]
    assert r.step == 4


def test_trainer_fits_from_a_replay_checkpoints_and_resumes(tmp_path):
    from tacorl_b200 import ops
    from tacorl_b200 import trainer as TR
    from tacorl_b200.replay import ReplayIndex
    ops.set_precision("fp32")
    T = 8
    ix = ReplayIndex(_episodes({"rgb_static": (84, 84)}, seed=7))

    def fresh():
        return _tacorl_module(T), _replay(ix, "tacorl", batch_size=3, min_window=4, max_window=T, pad=4)

    t, r = fresh()
    torch.manual_seed(1)
    tr = TR.Trainer(max_steps=5, precision="fp32", default_root_dir=tmp_path, steps_per_epoch=2)
    tr.fit(t, r)
    assert tr.global_step == 5 and t.current_epoch == 2 and r.step == 5
    assert len(tr.losses) == 5 and bool(torch.isfinite(torch.stack(tr.losses)).all())
    assert [o.steps_done for o in t.optimizers()] == [5] * len(t.optimizers())
    last = tmp_path / "saved_models" / "last.ckpt"
    assert last.is_file() and (tmp_path / "saved_models" / "tacorl_epoch_02_.ckpt").is_file()
    ck = torch.load(last, weights_only=False)
    assert ck["global_step"] == 5 and ck["replay"]["step"] == 5
    t2, r2 = fresh()
    tr2 = TR.Trainer(max_steps=7, precision="fp32", default_root_dir=tmp_path / "resumed", steps_per_epoch=2)
    tr2.fit(t2, r2, ckpt_path=last)
    assert tr2.global_step == 7 and r2.step == 7
    assert [o.steps_done for o in t2.optimizers()] == [7] * len(t2.optimizers())
    # default epoch length: valid window starts on the rank over the per-rank batch
    assert r.steps_per_epoch == len(ix.valid_starts(4)) // 3
    t3, r3 = fresh()
    tr3 = TR.Trainer(max_epochs=1, precision="fp32")
    tr3.fit(t3, r3)
    assert tr3.global_step == r3.steps_per_epoch and t3.current_epoch == 1


def test_trainer_refuses_a_replay_of_another_device_or_rank():
    from tacorl_b200 import trainer as TR
    from tacorl_b200.replay import ReplayIndex
    ix = ReplayIndex(_episodes({"rgb_static": (12, 12)}, seed=9))
    r = _replay(ix, "play_lmp", device="cuda:0")
    t = _play_module(8)
    other = TR.Trainer(max_steps=1, precision="fp32", device=torch.device("cuda", 1))
    with pytest.raises(ValueError, match="lives on cuda:0"):
        other.fit(t, r)
    wrong_rank = TR.Trainer(max_steps=1, precision="fp32", device=torch.device("cuda", 0))
    wrong_rank.world, wrong_rank.rank = 2, 1
    with pytest.raises(ValueError, match="shard 0 of 1"):
        wrong_rank.fit(t, r)


def test_replay_defaults_to_the_local_rank_device(monkeypatch):
    from tacorl_b200.replay import DeviceReplay, ReplayIndex
    monkeypatch.setenv("LOCAL_RANK", "0")
    ix = ReplayIndex(_episodes({"rgb_static": (12, 12)}, seed=9))
    r = DeviceReplay(ix, 4, min_window=2, max_window=4)
    assert r.device == torch.device("cuda", 0) and r.store["rgb_static"].device == torch.device("cuda", 0)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_ranks_get_disjoint_shards_and_their_own_draws():
    """Two ranks on cuda:0 and cuda:1, each sampling while the OTHER device is current: sample() launches on its own
    device's stream.  Shards are disjoint and cover the episodes; the ranks' draws differ and each equals the oracle's
    for its rank."""
    from tacorl_b200.replay import ReplayIndex
    eps = _episodes({"rgb_static": (12, 12)}, seed=8)
    reps = []
    for rank in range(2):
        ix = ReplayIndex(eps, rank=rank, world_size=2)
        with torch.cuda.device(1 - rank):
            reps.append(_replay(ix, "tacorl", device=f"cuda:{rank}", seed=5))
    a, b = (set(rp.index.episode_ids) for rp in reps)
    assert not a & b and a | b == set(range(len(LENGTHS)))
    tabs = []
    for rank, rp in enumerate(reps):
        with torch.cuda.device(1 - rank):
            rp.sample()
        torch.cuda.synchronize(rank)
        assert rp.tab.device == torch.device("cuda", rank) and rp.rank == rank
        assert np.array_equal(rp.tab.cpu().numpy(), _oracle_tables(rp, 0)["tab"])
        tabs.append(rp.shift.cpu().numpy())
    assert not np.array_equal(tabs[0], tabs[1])          # same seed, different ranks: different streams
