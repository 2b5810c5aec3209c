"""GPU tests of the per-step training metrics (DESIGN.md section 15): recorded rows against the values the modules
logged, epoch means against the rows, training unchanged by the record launch, no host sync between read-backs,
resume and two ranks."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.gpu_util import DEV
from tests.test_gpu_validation import _assert_same, _cpu, _episodes, _module, _opt_states, _train_replay

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def index84():
    from tacorl_b200.replay import ReplayIndex
    return ReplayIndex(_episodes({"rgb_static": (84, 84)}, seed=5))


@pytest.fixture
def logged_after_each_step(monkeypatch):
    """Collects {key: float32 value} of every `train/*` tensor in module.logged right after each step (a host sync,
    which only the test makes) by hooking the recorder's host-side step_done."""
    from tacorl_b200 import runtime
    seen = []
    state = {"module": None}
    orig = runtime.TrainMetricsRecorder.step_done

    def step_done(self, global_step, epoch):
        torch.cuda.synchronize()
        vals = {k: np.float32(v.float().item()) for k, v in state["module"].logged.items()
                if k.startswith("train/") and torch.is_tensor(v)}
        seen.append((global_step, epoch, vals))
        orig(self, global_step, epoch)
    monkeypatch.setattr(runtime.TrainMetricsRecorder, "step_done", step_done)
    return seen, state


def _bits(x):
    return np.asarray(x, np.float32).view(np.int32)


def _check_epoch_means(tr):
    """Each epoch mean equals the step-ordered fp64 sum of its recorded rows over their count, bit for bit."""
    h = tr.train_history
    vals, epochs = h.values, h.epochs
    for epoch, _, means in tr.train_epoch_history:
        rows = vals[epochs == epoch]
        want = {}
        for i, k in enumerate(h.keys):
            s, n = 0.0, 0
            for v in rows[:, i]:
                if not np.isnan(v):
                    s += float(v)
                    n += 1
            if n:
                want[k] = s / n
        assert means == want, (epoch, means, want)


@pytest.mark.parametrize("graphed", [True, False], ids=["graph", "eager"])
@pytest.mark.parametrize("fed", ["host", "replay"])
@pytest.mark.parametrize("kind", ["play_lmp", "tacorl", "cql"])
def test_recorded_rows_are_the_logged_values_and_epoch_means_their_fp64_means(index84, logged_after_each_step, kind,
                                                                              fed, graphed):
    from tacorl_b200 import trainer as TR
    seen, state = logged_after_each_step
    m = state["module"] = _module(kind, bc_epochs=1)       # TACO-RL crosses bc_epochs after the first epoch
    train = _train_replay(index84, kind)
    torch.manual_seed(1)
    tr = TR.Trainer(max_steps=8, precision="fp32", steps_per_epoch=3, log_every_n_steps=2, use_cuda_graph=graphed)
    if fed == "host":
        hosts = [_cpu(train.sample()) for _ in range(3)]
        tr.fit(m, lambda s: hosts[s % 3])
    else:
        tr.fit(m, train)
    h = tr.train_history
    assert len(h) == 8 and h.steps.tolist() == list(range(8))
    assert h.epochs.tolist() == [0, 0, 0, 1, 1, 1, 2, 2]
    assert [(g, e) for g, e, _ in seen] == list(zip(range(8), [0, 0, 0, 1, 1, 1, 2, 2]))
    assert set(h.keys) == set().union(*[v.keys() for _, _, v in seen]) and len(h.keys) >= 2
    vals = h.values
    for j, (_, _, logged) in enumerate(seen):
        for i, k in enumerate(h.keys):
            want = logged.get(k, np.float32("nan"))
            assert _bits(vals[j, i]) == _bits(want), (kind, j, k, vals[j, i], want)
    assert [(e, s) for e, s, _ in tr.train_epoch_history] == [(0, 3), (1, 6)]
    assert tr.train_epoch_metrics == tr.train_epoch_history[-1][2]
    assert set(tr.train_epoch_metrics) == set(h.keys)
    _check_epoch_means(tr)
    if graphed:
        assert tr._train_graph.captures == (2 if kind == "tacorl" else 1)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["play_lmp", "tacorl", "cql"])
def test_recording_leaves_training_unchanged_and_adds_one_launch(index84, kind, precision):
    from tacorl_b200 import ops, runtime
    from tacorl_b200 import trainer as TR
    n = 5

    m = _module(kind, precision)
    train = _train_replay(index84, kind)
    torch.manual_seed(1)
    tr = TR.Trainer(max_steps=n, precision=precision, steps_per_epoch=100, log_every_n_steps=2)
    tr.fit(m, train)
    got = ({k: v.detach().cpu().clone() for k, v in m.state_dict().items()}, _opt_states(m))
    assert len(tr.train_history) == n

    p = _module(kind, precision)
    plain = _train_replay(index84, kind)
    ops.set_precision(precision)
    p.train()
    opts = TR._optimizers_of(p)
    fn = runtime.play_lmp_step_fn(p, opts[0]) if kind == "play_lmp" else runtime.tacorl_step_fn(p)
    torch.manual_seed(1)
    g = runtime.GraphedTrainStep(fn, None, device=torch.device(DEV, 0), warmup=2, source=plain)
    for _ in range(n):
        g()
    torch.cuda.synchronize()
    want = ({k: v.detach().cpu().clone() for k, v in p.state_dict().items()}, _opt_states(p))
    assert train.step == plain.step == n
    _assert_same(got[0], want[0], "state_dict")
    _assert_same(got[1], want[1], "optimizer_states")
    assert tr._train_graph.launches_per_replay == g.launches_per_replay + 1


def test_no_host_sync_between_read_backs_and_one_side_stream_copy_per_half(index84, tmp_path):
    from torch.profiler import ProfilerActivity, profile, record_function

    from tacorl_b200 import trainer as TR
    every = 4
    m = _module("play_lmp")
    train = _train_replay(index84, "play_lmp")
    batches = [_clone(train.sample()) for _ in range(2)]          # device batches: no host-to-device copy
    prof = profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA])

    def get(s):
        if s == 1:                       # step 0 captured the graph; steps 1 .. 2 * every only replay it
            torch.cuda.synchronize()
            prof.start()
        elif s == 1 + 2 * every:
            with record_function("test_drain"):
                torch.cuda.synchronize()
            prof.stop()
        return batches[s % 2]
    tr = TR.Trainer(max_steps=2 * every + 2, precision="fp32", log_every_n_steps=every, default_root_dir=tmp_path)
    tr.fit(m, get)
    trace = tmp_path / "trace.json"
    prof.export_chrome_trace(str(trace))
    events = [e for e in json.loads(trace.read_text())["traceEvents"] if e.get("ph") == "X"]
    drain = [e for e in events if e["name"] == "test_drain"]
    assert len(drain) == 1
    syncs = [e["name"] for e in events if "Synchronize" in e["name"] and e["ts"] < drain[0]["ts"]]   # the steps ran before
    assert not syncs, syncs
    record = {e["args"]["stream"] for e in events if e.get("cat") == "kernel" and "metrics_record" in e["name"]}
    assert len(record) == 1                               # the training stream
    d2h = [e for e in events if e.get("cat") == "gpu_memcpy" and "DtoH" in e["name"]]
    assert len(d2h) == 2, [e["name"] for e in d2h]        # steps every - 1 and 2 * every - 1 finished a half each
    assert all(e["args"]["stream"] not in record for e in d2h)
    assert not [e for e in events if e.get("cat") == "gpu_memcpy" and "HtoD" in e["name"]]
    assert len(tr.train_history) == 2 * every + 2


def _clone(batch):
    return {k: _clone(v) if isinstance(v, dict) else v.clone() for k, v in batch.items()}


def _csv_rows(path):
    import csv
    text = path.read_text()
    with open(path, newline="") as f:
        return text, list(csv.DictReader(f))


def test_resume_restores_the_epoch_history_and_appends_to_metrics_csv(index84, tmp_path):
    from tacorl_b200 import trainer as TR
    k, every = 5, 2
    m, train = _module("tacorl", bc_epochs=1), _train_replay(index84, "tacorl")
    torch.manual_seed(1)
    tr1 = TR.Trainer(max_steps=k, precision="fp32", default_root_dir=tmp_path, steps_per_epoch=3,
                     log_every_n_steps=every)
    tr1.fit(m, train)
    last = tmp_path / "saved_models" / "last.ckpt"
    ck = torch.load(last, weights_only=False)
    assert ck["training"]["epoch_history"] == tr1.train_epoch_history and len(tr1.train_epoch_history) == 1
    assert ck["training"]["metrics"] == tr1.train_epoch_metrics
    assert tr1.train_history.steps.tolist() == list(range(k))

    m2, train2 = _module("tacorl", bc_epochs=1), _train_replay(index84, "tacorl")
    torch.manual_seed(2)
    tr2 = TR.Trainer(max_steps=2 * k, precision="fp32", default_root_dir=tmp_path, steps_per_epoch=3,
                     log_every_n_steps=every)
    tr2.fit(m2, train2, ckpt_path=last)
    assert tr2.train_epoch_history[:1] == ck["training"]["epoch_history"]
    assert [(e, s) for e, s, _ in tr2.train_epoch_history] == [(0, 3), (1, 8)]   # the resumed epoch runs 3 more steps
    h = tr2.train_history
    assert h.steps.tolist() == list(range(k, 2 * k))
    assert h.epochs.tolist() == [ck["epoch"]] * 3 + [ck["epoch"] + 1] * 2
    text, rows = _csv_rows(tmp_path / "metrics.csv")
    assert text.count("step,epoch") == 1
    keys = [c for c in rows[0] if c not in ("step", "epoch") and not c.endswith("_epoch")]
    step_rows = [r for r in rows if any(r[c] for c in keys)]
    epoch_rows = [r for r in rows if not any(r[c] for c in keys)]
    assert [int(r["step"]) for r in step_rows] == [s for s in range(2 * k) if (s + 1) % every == 0]
    assert [(int(r["step"]), int(r["epoch"])) for r in epoch_rows] == [(2, 0), (7, 1)]
    by_step = {int(r["step"]): r for r in step_rows}
    for s in (5, 7, 9):
        j = s - k
        for i, key in enumerate(h.keys):
            assert float(by_step[s][key]) == float(h.values[j, i]) or np.isnan(h.values[j, i])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_ranks_record_the_mean_over_ranks_on_both(tmp_path):
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr=127.0.0.1", "--master-port=29533",
           os.path.join(ROOT, "tests", "workers", "train_metrics_worker.py"), str(tmp_path)]
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    out = [json.loads((tmp_path / f"rank{r}.json").read_text()) for r in range(2)]
    assert out[0]["keys"] == out[1]["keys"] and out[0]["steps"] == out[1]["steps"]
    rows = [np.asarray(o["rows"], np.float32) for o in out]
    assert np.array_equal(_bits(rows[0]), _bits(rows[1]))
    logged = [np.asarray(o["logged"], np.float32) for o in out]
    assert not np.array_equal(logged[0], logged[1])          # the ranks train on different shards
    want = (logged[0] + logged[1]) / np.float32(2)
    assert np.array_equal(_bits(rows[0]), _bits(want))
    assert out[0]["epoch_metrics"] == out[1]["epoch_metrics"]
