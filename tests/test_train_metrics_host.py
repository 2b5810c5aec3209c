"""Host tests of the training-metrics recorder's bookkeeping (DESIGN.md section 15): ring rows and halves, the step
mapping across a mid-interval resume, epoch means with per-key counts, rank combination, metrics.csv and the key
limit.  No GPU needed."""
import csv
import math

import numpy as np
import pytest

from tacorl_b200 import runtime as R

M = 32


def _drive(book, first_step, n, epoch_of=lambda s: 0):
    takes = []
    for s in range(first_step, first_step + n):
        got = book.advance(s, epoch_of(s))
        if got is not None:
            takes.append(got)
    return takes


def test_ring_rows_halves_and_a_flush_in_the_middle_of_a_half():
    book = R.RingBook(3)                                  # ring of 6 rows
    takes = _drive(book, 0, 7)
    assert [(t[0], t[1].tolist()) for t in takes] == [(0, [0, 1, 2]), (3, [3, 4, 5])]
    flushed = book.take()                                 # epoch end after step 6: row 0, the third half's start
    assert flushed[0] == 0 and flushed[1].tolist() == [6]
    assert book.take() is None
    takes = _drive(book, 7, 5)                            # the rest of that half, then the next one
    assert [(t[0], t[1].tolist()) for t in takes] == [(1, [7, 8]), (3, [9, 10, 11])]
    for row0, steps, _ in takes + [flushed]:
        assert row0 // 3 == (row0 + len(steps) - 1) // 3      # a range never spans two halves


def test_a_resume_in_the_middle_of_an_interval_maps_rows_to_global_steps():
    every = 4
    book = R.RingBook(every)
    takes = _drive(book, 10, 9, epoch_of=lambda s: s // 6)     # resumed at global step 10, 6 steps an epoch
    takes.append(book.take())
    steps = np.concatenate([t[1] for t in takes])
    epochs = np.concatenate([t[2] for t in takes])
    assert steps.tolist() == list(range(10, 19))
    assert epochs.tolist() == [s // 6 for s in range(10, 19)]
    assert [t[0] for t in takes] == [0, 4, 0]                 # rows count from the resume, not from step 0
    rows = []
    for _, st, ep in takes:
        vals = st[:, None].astype(np.float32) * np.ones((1, 2), np.float32)
        rows += R.logging_rows(["train/a", "train/b"], st, ep, vals, every)
    assert [(r["step"], r["epoch"]) for r in rows] == [(11, 1), (15, 2)]    # (step + 1) % 4 == 0
    assert rows[0]["train/a"] == 11.0


def _acc(values):
    """The recorder's fp64 (sums, counts) vector after recording `values` (one list per step, None = not logged)."""
    acc = [0.0] * (2 * M)
    for row in values:
        for i, v in enumerate(row):
            if v is not None:
                acc[i] += float(np.float32(v))
                acc[M + i] += 1.0
    return acc


def test_epoch_means_count_each_key_over_the_steps_that_logged_it():
    keys = R.assign_columns([], ["train/q1_loss"])
    steps = [[0.5], [0.25]]                                  # BC epoch: one key
    R.assign_columns(keys, ["train/q1_loss", "train/actor_loss"])
    steps += [[0.125, 2.0], [1.0, 4.0], [3.0, 8.0]]          # the Q mode adds a key mid-epoch
    means = R.epoch_means(keys, [_acc(steps)])
    assert keys == ["train/q1_loss", "train/actor_loss"]
    assert means["train/q1_loss"] == (0.5 + 0.25 + 0.125 + 1.0 + 3.0) / 5
    assert means["train/actor_loss"] == (2.0 + 4.0 + 8.0) / 3
    assert R.epoch_means(keys + ["train/never"], [_acc(steps)]).keys() == means.keys()   # no step: no mean
    with pytest.raises(ValueError):
        R.epoch_means(keys, [[0.0] * M])


def test_ranks_are_summed_before_dividing():
    keys = ["train/x", "train/y"]
    r0 = _acc([[1.0, None], [2.0, 5.0]])
    r1 = _acc([[10.0, 7.0]])
    means = R.epoch_means(keys, [r0, r1])
    assert means == {"train/x": 13.0 / 3, "train/y": 12.0 / 2}


def test_train_history_keeps_rows_and_pads_keys_a_later_block_added():
    h = R.TrainHistory()
    h.append(["train/a"], [0, 1], [0, 0], np.array([[1.0, 9.0], [2.0, 9.0]], np.float32))   # ring columns: 2
    h.append(["train/a", "train/b"], [2], [1], np.array([[3.0, 4.0]], np.float32))
    assert len(h) == 3 and h.keys == ["train/a", "train/b"]
    assert h.steps.tolist() == [0, 1, 2] and h.epochs.tolist() == [0, 0, 1]
    v = h.values
    assert v.dtype == np.float32 and v[:, 0].tolist() == [1.0, 2.0, 3.0]
    assert math.isnan(v[0, 1]) and math.isnan(v[1, 1]) and v[2, 1] == 4.0
    assert h.column("train/b")[2] == 4.0


def _read(path):
    with open(path, newline="") as f:
        text = f.read()
    with open(path, newline="") as f:
        return text, list(csv.DictReader(f))


def test_metrics_csv_layout_and_appending_on_resume(tmp_path):
    path = tmp_path / "metrics.csv"
    w = R.MetricsCSV(path, 0)
    w.write([{"step": 1, "epoch": 0, "train/a": 0.5}, {"step": 3, "epoch": 0, "train/a": 0.25}])
    w.write([{"step": 3, "epoch": 0, "train/a_epoch": 0.375}])
    w.write([{"step": 5, "epoch": 1, "train/a": 1.5, "train/b": float("nan")}])   # a new key widens the header
    text, rows = _read(path)
    assert text.splitlines()[0] == "step,epoch,train/a,train/b,train/a_epoch,train/b_epoch"
    assert text.count("step,epoch") == 1
    assert [(r["step"], r["train/a"], r["train/a_epoch"]) for r in rows] == [
        ("1", "0.5", ""), ("3", "0.25", ""), ("3", "", "0.375"), ("5", "1.5", "")]
    assert rows[3]["train/b"] == "nan"
    # resume from a checkpoint at global step 4: the row of step 5 came after it and goes
    w2 = R.MetricsCSV(path, 4)
    w2.write([{"step": 5, "epoch": 1, "train/a": 2.5, "train/b": 1.0}, {"step": 7, "epoch": 1, "train/b": 3.0}])
    text, rows = _read(path)
    assert text.count("step,epoch") == 1
    assert [r["step"] for r in rows] == ["1", "3", "3", "5", "7"]
    assert rows[3]["train/a"] == "2.5" and rows[4]["train/a"] == "" and rows[4]["train/b"] == "3.0"
    # a run from step 0 into the same directory starts the file over
    R.MetricsCSV(path, 0)
    assert _read(path)[1] == []


def test_more_than_32_keys_are_refused_and_columns_keep_first_appearance_order():
    keys = R.assign_columns([], [f"train/k{i}" for i in range(20)])
    R.assign_columns(keys, ["train/k3", "train/new"] + [f"train/k{i}" for i in range(20)])
    assert keys[:20] == [f"train/k{i}" for i in range(20)] and keys[20] == "train/new"
    R.assign_columns(keys, [f"train/m{i}" for i in range(11)])
    assert len(keys) == 32
    with pytest.raises(ValueError, match="more than 32"):
        R.assign_columns(keys, ["train/one_more"])


def test_log_every_n_steps_must_be_positive():
    from tacorl_b200 import trainer as TR
    assert TR.Trainer().log_every_n_steps == 50
    with pytest.raises(ValueError, match="log_every_n_steps"):
        TR.Trainer(log_every_n_steps=0)
