"""Long chains through the persistent recurrence kernels: the per-step hand-off (arrival counters, per-K-block operand
loads, the cluster reduction) has to hold over many phases, not only the 16 steps of test_gpu_rnn_bf16_oracle.py.

Each case runs tacorl_rnn_layer2_fwd / _bwd with seq_enable = 1 (persistent), 0 (per-step launches) and, with two
directions, 2 (the two lanes launched one after the other).  Asserted: the persistent run is within the oracle's
tolerance (tests/rnn_bf16_oracle.py) forward and backward; two lanes in one launch equal two one-lane launches bit for
bit; seq8 (batch 65..128) equals the per-step path bit for bit; no flag wait timed out."""
import pytest

from tests.test_gpu_rnn_bf16_oracle import Layer2, _same

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L():
    from tacorl_b200 import _lib
    lib = _lib.lib()
    was = lib.tacorl_rnn_seq_enable(1)
    yield _lib
    lib.tacorl_rnn_seq_enable(was)
    assert lib.tacorl_rnn_seq_timeouts() == 0      # (synchronises the device)


def _run(L, c, modes):
    lib = L.lib()
    runs = {}
    try:
        for mode in modes:
            lib.tacorl_rnn_seq_enable(mode)
            f = c.fwd(L)
            runs[mode] = (f, c.bwd(L, runs[1][0] if 1 in runs else f))   # every BPTT on the mode-1 forward
    finally:
        lib.tacorl_rnn_seq_enable(1)
    return runs


WAVE_CASES = [(T, B, H, D) for T in (64, 97) for B in (3, 17, 63, 64) for H in (256, 2048) for D in (1, 2)]


@pytest.mark.parametrize("case", WAVE_CASES, ids=lambda c: "T{}B{}H{}D{}".format(*c))
def test_wave_chain(L, case):
    T, B, H, D = case
    c = Layer2(T, B, 32, H, D, T, 0, 1, seed=T * 1000 + B * 7 + H + D)
    runs = _run(L, c, [1, 0, 2] if D == 2 else [1, 0])
    f1, b1 = runs[1]
    f0, b0 = runs[0]
    # persistent: the per-step path launches at least once per step, each way
    assert f1["launches"] + T // 2 <= f0["launches"] and b1["launches"] + T // 2 <= b0["launches"]
    c.check_fwd(f1, "persistent")
    c.check_bwd(f1, b1, "persistent")
    if D == 2:
        f2, b2 = runs[2]
        assert f2["launches"] == f1["launches"] + 1
        for k in ("out", "outb"):
            assert _same(f2[k], f1[k]), k
        for k in ("dpre", "dpb", "dx"):
            assert _same(b2[k], b1[k]), k
        assert all(_same(u, v) for u, v in zip(b2["dw"], b1["dw"]))
    assert L.lib().tacorl_rnn_seq_timeouts() == 0


@pytest.mark.parametrize("B", [65, 128])
def test_seq8_chain_bit_identical_to_per_step(L, B):
    T, H = 64, 2048
    c = Layer2(T, B, 32, H, 1, 0, 0, 1, seed=B)
    runs = _run(L, c, [1, 0])
    f1, b1 = runs[1]
    f0, b0 = runs[0]
    assert f1["launches"] + T // 2 <= f0["launches"] and b1["launches"] + T // 2 <= b0["launches"]
    c.check_fwd(f1, "seq8")
    c.check_bwd(f1, b1, "seq8")
    for k in ("out", "outb"):
        assert _same(f1[k], f0[k]), k
    for k in ("dpre", "dpb", "dx"):
        assert _same(b1[k], b0[k]), k
    assert L.lib().tacorl_rnn_seq_timeouts() == 0
