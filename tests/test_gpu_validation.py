"""GPU tests of validation sweeps (DESIGN.md section 14): the sweep-mode sampler and gather against the numpy
restatement (tests/sweep_oracle.py), Trainer.validate against eager validation_step calls, and fit(val=) against fit
without validation."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import replay_oracle as RO
from oracle import synth as S
from tests import sweep_oracle as SO
from tests.gpu_util import DEV, build_cql_flat, build_play_lmp, build_tacorl

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LENGTHS = [12, 5, 30, 1, 9, 3, 20, 2, 17]
T = 8


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


def _sweep_replay(index, kind, B, **kw):
    from tacorl_b200.replay import DeviceReplay
    args = dict(batch_size=B, kind=kind, min_window=4, max_window=T, goal_p=0.3, neg_frac=0.25, seed=11, device=DEV,
                mode="sweep")
    args.update(kw)
    return DeviceReplay(index, **args)


def _train_replay(index, kind, B=3):
    from tacorl_b200.replay import DeviceReplay
    return DeviceReplay(index, B, kind=kind, min_window=4, max_window=T, pad=4, seed=3, device=DEV)


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


def _module(kind, precision="fp32", bc_epochs=0):
    if kind == "cql":
        m = build_cql_flat(precision)
        seed = 29
    else:
        lmp = build_play_lmp("tanh_net", ("rgb_static",), 128, 16, T)
        m = lmp if kind == "play_lmp" else build_tacorl(lmp, precision, bc_epochs=bc_epochs)
        seed = 4 if kind == "play_lmp" else 6
    shapes = {k: list(v.shape) for k, v in m.state_dict().items()}
    m.load_state_dict(S.synth_state_dict(shapes, seed))
    m.to(DEV)
    m.train()
    m.optimizers()
    return m


@pytest.fixture(scope="module")
def two_view_index():
    from tacorl_b200.replay import ReplayIndex
    return ReplayIndex(_episodes({"rgb_static": (24, 36), "rgb_gripper": (12, 12)}),
                       modalities=("rgb_static", "rgb_gripper"))


@pytest.fixture(scope="module")
def index84():
    from tacorl_b200.replay import ReplayIndex
    return ReplayIndex(_episodes({"rgb_static": (84, 84)}, seed=5))


@pytest.mark.parametrize("kind", ["play_lmp", "tacorl", "cql"])
def test_sweep_tables_and_batches_equal_the_oracle_for_full_batches_and_the_tail(two_view_index, kind):
    ix = two_view_index
    r = _sweep_replay(ix, kind, 16, min_window=2)
    assert r.tail and r.batches_per_sweep >= 2 and r.items == len(ix.items(kind, 2))
    want = SO.sweep(kind, ix, 16, r.seed, min_window=2, max_window=T, goal_p=0.3, neg_frac=0.25)
    for rep in range(2):                              # two sweeps: the same tables
        r.reset()
        for t in want:
            n = t["tab"].shape[1]
            got = _cpu(r.sample(n))
            assert np.array_equal(r.tab[:, :n].cpu().numpy(), t["tab"]), (kind, rep, n)
            assert np.array_equal(r.out64[:, :n].cpu().numpy(), t["out64"]), (kind, rep, n)
            _assert_batches_equal(got, RO.assemble(kind, t, ix.frames, ix.actions, r.T, 0, list(ix.modalities)))
        assert int(r.preserve()[0].item()) == r.items
    with pytest.raises(ValueError):
        r.sample(17)


def _eager_means(module, val, seed):
    """Item-weighted means of eager validation_step calls over the sweep's batches, in eval mode."""
    flags = [(m, m.training) for m in module.modules()]
    module.eval()
    torch.cuda.manual_seed(seed)
    val.reset()
    sums, count = {}, 0
    for n in [val.B] * val.batches_per_sweep + ([val.tail] if val.tail else []):
        batch = val.sample(n)
        with torch.no_grad():
            module.validation_step(batch, 0)
        for k, v in module.logged.items():
            if k.startswith("validation/"):
                sums[k] = sums.get(k, 0.0) + n * float(v)
        count += n
    for m, t in flags:
        m.training = t
    return {k: v / count for k, v in sums.items()}, count


def _assert_metrics_close(got, want, rtol=1e-6):
    assert set(got) == set(want), set(got) ^ set(want)
    for k in want:
        assert abs(got[k] - want[k]) <= rtol * abs(want[k]) + 1e-9, (k, got[k], want[k])


@pytest.mark.parametrize("kind", ["play_lmp", "tacorl", "cql"])
def test_validate_equals_the_item_weighted_mean_of_eager_validation_steps(index84, kind):
    from tacorl_b200 import trainer as TR
    m = _module(kind)
    val = _sweep_replay(index84, kind, 7)
    assert val.tail and val.batches_per_sweep >= 2
    tr = TR.Trainer(precision="fp32")
    [got] = tr.validate(m, val)
    assert m.training and tr.callback_metrics == got
    want, count = _eager_means(m, val, TR.VALIDATION_SEED)
    assert count == val.items
    _assert_metrics_close(got, want)
    [again] = tr.validate(m, val)                      # the same weights: bit-identical
    assert again == got


def _opt_states(m):
    from tacorl_b200.trainer import _optimizers_of
    return [o.state_dict() for o in _optimizers_of(m)]


def _assert_same(a, b, path=""):
    if torch.is_tensor(a):
        assert torch.equal(a.cpu(), b.cpu()), path
    elif isinstance(a, dict):
        assert set(a) == set(b), path
        for k in a:
            _assert_same(a[k], b[k], f"{path}.{k}")
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            _assert_same(x, y, f"{path}[{i}]")
    else:
        assert a == b, path


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["play_lmp", "tacorl", "cql"])
def test_fit_with_validation_trains_bit_for_bit_like_fit_without(index84, kind, precision):
    from tacorl_b200 import trainer as TR

    def run(with_val):
        m = _module(kind, precision, bc_epochs=1)      # TACO-RL crosses bc_epochs after the first epoch
        train = _train_replay(index84, kind)
        val = _sweep_replay(index84, kind, 4) if with_val else None
        torch.manual_seed(1)
        tr = TR.Trainer(max_epochs=3, precision=precision, steps_per_epoch=2)
        tr.fit(m, train, val=val)
        sd = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
        return sd, _opt_states(m), train.step, m, tr

    sd0, opt0, step0, _, _ = run(False)
    sd1, opt1, step1, m1, tr1 = run(True)
    assert step0 == step1 == 6
    _assert_same(sd1, sd0, "state_dict")
    _assert_same(opt1, opt0, "optimizer_states")
    assert m1.training
    assert [(e, s) for e, s, _ in tr1.val_history] == [(0, 2), (1, 4), (2, 6)]
    assert all(np.isfinite(v) for _, _, mt in tr1.val_history for v in mt.values())
    assert tr1.callback_metrics == tr1.val_history[-1][2]


def test_validation_graph_adds_three_launches_and_a_sweep_copies_once_to_the_host(index84):
    from torch.profiler import ProfilerActivity, profile

    from tacorl_b200 import _lib
    from tacorl_b200 import trainer as TR
    m = _module("play_lmp")
    val = _sweep_replay(index84, "play_lmp", 4)
    assert val.tail
    tr = TR.Trainer(precision="fp32")
    tr.validate(m, val)
    graph = tr._val_states[(id(m), id(val))]["graph"]
    m.eval()
    batch = val.sample()
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with torch.no_grad():
        m.validation_step(batch, 0)
    forward = _lib.launch_count() - n0
    m.train()
    assert graph.launches_per_replay == forward + 3          # sweep, gather, accumulate
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        tr.validate(m, val)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert not [n for n in names if "HtoD" in n or "Host to Device" in n], sorted(set(names))[:40]
    assert len([n for n in names if "DtoH" in n or "Device to Host" in n]) == 1, \
        [n for n in names if "Memcpy" in n or "memcpy" in n]


def test_resume_from_a_checkpoint_written_with_validation(index84, tmp_path):
    from tacorl_b200 import trainer as TR
    ckpts = {}
    for name, with_val in (("val", True), ("plain", False)):
        m, train = _module("tacorl", bc_epochs=1), _train_replay(index84, "tacorl")
        torch.manual_seed(1)
        tr = TR.Trainer(max_steps=4, precision="fp32", default_root_dir=tmp_path / name, steps_per_epoch=2)
        tr.fit(m, train, val=_sweep_replay(index84, "tacorl", 4) if with_val else None)
        ckpts[name] = tmp_path / name / "saved_models" / "last.ckpt"
    ck = torch.load(ckpts["val"], weights_only=False)
    plain = torch.load(ckpts["plain"], weights_only=False)
    assert "validation" not in plain
    assert [(e, s) for e, s, _ in ck["validation"]["history"]] == [(0, 2), (1, 4)]
    assert ck["validation"]["metrics"] == ck["validation"]["history"][-1][2]
    assert torch.load(tmp_path / "val" / "saved_models" / "tacorl_epoch_01_.ckpt",
                      weights_only=False)["validation"]["history"][0][:2] == (0, 2)
    _assert_same(ck["state_dict"], plain["state_dict"], "state_dict")
    finals = {}
    for name in ("val", "plain"):
        m, train = _module("tacorl", bc_epochs=1), _train_replay(index84, "tacorl")
        val = _sweep_replay(index84, "tacorl", 4)
        torch.manual_seed(2)
        tr = TR.Trainer(max_steps=8, precision="fp32", steps_per_epoch=2)
        tr.fit(m, train, ckpt_path=ckpts[name], val=val)
        assert tr.global_step == 8 and train.step == 8 and m.current_epoch == 4
        finals[name] = ({k: v.detach().cpu().clone() for k, v in m.state_dict().items()}, _opt_states(m),
                        [h[:2] for h in tr.val_history], tr.val_history[-1][2])
    _assert_same(finals["val"][0], finals["plain"][0], "state_dict")
    _assert_same(finals["val"][1], finals["plain"][1], "optimizer_states")
    assert finals["val"][2] == [(0, 2), (1, 4), (2, 6), (3, 8)]
    assert finals["plain"][2] == [(2, 6), (3, 8)]
    assert finals["val"][3] == finals["plain"][3]


@pytest.mark.parametrize("kind", ["play_lmp", "cql"])
def test_host_batch_validation_matches_the_replay_sweep(index84, kind):
    from tacorl_b200 import trainer as TR
    m = _module(kind)
    val = _sweep_replay(index84, kind, 7)
    assert val.tail
    host = []
    val.reset()
    for n in [val.B] * val.batches_per_sweep + [val.tail]:
        host.append(_cpu(val.sample(n)))
    tr = TR.Trainer(precision="fp32")
    [from_host] = tr.validate(m, host)
    [from_replay] = tr.validate(m, val)
    _assert_metrics_close(from_host, from_replay)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_ranks_with_unequal_items_give_the_item_mean_over_both_shards(tmp_path):
    from tacorl_b200 import trainer as TR
    from tacorl_b200.replay import ReplayIndex
    out = tmp_path / "metrics.json"
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr=127.0.0.1", "--master-port=29531", os.path.join(ROOT, "tests", "workers", "validation_worker.py"),
           str(out)]
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    got = json.loads(out.read_text())
    from tests.workers.validation_worker import episodes, shard_replay
    sums, count = {}, 0
    for rank in range(2):
        val = shard_replay(ReplayIndex(episodes(), rank=rank, world_size=2), DEV)
        means, n = _eager_means(_module("play_lmp"), val, TR.VALIDATION_SEED)
        for k, v in means.items():
            sums[k] = sums.get(k, 0.0) + n * v
        count += n
    assert got["items"][0] != got["items"][1]
    _assert_metrics_close(got["metrics"], {k: v / count for k, v in sums.items()})
