"""The teacher-forced bf16 RNN oracle (tests/rnn_bf16_oracle.py) checked on the CPU before any GPU is involved: a
torch emulation of the kernels' arithmetic (bf16 operands, fp32 accumulation, one step after another) passes the
check at the tolerance the GPU tests use, and every discrimination control fails it by at least 20x that tolerance."""
import pytest
import torch

from tests import rnn_bf16_oracle as R
from tests.rnn_bf16_oracle import TAU


def _bf(t):
    return t.bfloat16().float()


def emulate_fwd(x, w_ih, w_hh, b_ih, b_hh, h0, reverse, n):
    T, B, _ = x.shape
    H = w_hh.shape[0]
    out = torch.full((T, B, H), float("nan"))
    a = R.active(T, n, reverse)
    out[a] = _bf(x[a]) @ _bf(w_ih).t() + (b_ih + b_hh)
    prev = None if h0 is None else _bf(h0)
    for t in (range(T - 1, T - n - 1, -1) if reverse else range(n)):
        if prev is not None:
            out[t] = out[t] + prev @ _bf(w_hh).t()
        out[t] = torch.relu(out[t])
        prev = _bf(out[t])
    return out


def emulate_bwd(x, w_ih, w_hh, h0, out, dout, dhn, reverse, n):
    T, B, _ = x.shape
    a = R.active(T, n, reverse)
    dpre = dout.clone()
    carry = dhn
    for t in (range(T - n, T) if reverse else range(n - 1, -1, -1)):
        v = dpre[t] + carry if carry is not None else dpre[t]
        dpre[t] = v * (out[t] > 0)
        carry = _bf(dpre[t]) @ _bf(w_hh)
    db = _bf(dpre[a])
    hb = _bf(out)
    first = _bf(h0).unsqueeze(0) if h0 is not None else torch.zeros_like(hb[:1])
    hp = torch.cat([hb[T - n + 1:], first]) if reverse else torch.cat([first, hb[:n - 1]])
    flat = lambda t: t.reshape(-1, t.shape[-1])   # noqa: E731
    return {"dpre": dpre[a], "dw_hh": flat(db).t() @ flat(hp), "dw_ih": flat(db).t() @ flat(_bf(x[a])),
            "db": flat(dpre[a]).sum(0), "dx": db @ _bf(w_ih), "dh0": (db[-1] if reverse else db[0]) @ _bf(w_hh)}


def _case(T, B, I, H, seed, with_h0, with_dhn):
    g = torch.Generator().manual_seed(seed)
    k = 1.0 / H ** 0.5
    u = lambda *s: (torch.rand(*s, generator=g) * 2 - 1) * k   # noqa: E731  (nn.RNN's initialisation)
    x = torch.randn(T, B, I, generator=g)
    w_ih, w_hh, b_ih, b_hh = u(H, I), u(H, H), u(H), u(H)
    h0 = torch.rand(B, H, generator=g) if with_h0 else None
    dout = torch.randn(T, B, H, generator=g)
    dhn = torch.randn(B, H, generator=g) if with_dhn else None
    return x, w_ih, w_hh, b_ih, b_hh, h0, dout, dhn


@pytest.mark.parametrize("T,B,I,H,reverse,n", [(7, 24, 33, 512, False, 7), (7, 24, 33, 512, True, 4),
                                                (5, 3, 12, 256, True, 5), (9, 16, 48, 256, False, 1)])
def test_emulated_kernel_passes_and_controls_fail(T, B, I, H, reverse, n):
    x, w_ih, w_hh, b_ih, b_hh, h0, dout, dhn = _case(T, B, I, H, T * B + I + H, True, True)
    out = emulate_fwd(x, w_ih, w_hh, b_ih, b_hh, h0, reverse, n)
    got = emulate_bwd(x, w_ih, w_hh, h0, out, dout, dhn, reverse, n)
    got["out"] = out[R.active(T, n, reverse)]
    dpre_k = dout.clone()
    dpre_k[R.active(T, n, reverse)] = got["dpre"]

    def oracle(control=None):
        ref = R.fwd(x, w_ih, w_hh, b_ih, b_hh, out, h0, reverse, n, control)
        ref.update(R.bwd(x, w_ih, w_hh, out, dout, dpre_k, h0, dhn, reverse, n, control))
        return ref

    ref = oracle()
    res = R.check_all(got, ref, TAU)
    assert all(r[0] for r in res.values()), {k: r[1] for k, r in res.items()}
    # the emulation is much closer than TAU: the bar has head room for the kernels' own summation orders
    assert max(r[1] for r in res.values()) < TAU / 4, {k: r[1] for k, r in res.items()}
    for control in R.CONTROLS:
        if control in ("fp32_hidden", "shift_pairs") and n == 1:
            continue     # a single step consumes no hidden state of its own and has no pairs
        res = R.check_all(got, oracle(control), TAU)
        worst = max(r[1] for r in res.values())
        assert worst >= 20 * TAU, (control, {k: r[1] for k, r in res.items()})
    for name in ("out", "dpre", "dw_hh", "dw_ih", "db", "dx", "dh0"):
        want, scale = ref[name]
        ok, ratio, _, _ = R.check(R.bump_one_ulp(got[name], want, scale), want, scale, TAU)
        assert not ok and ratio >= 20 * TAU, (name, ratio)


def test_check_reports_per_step_errors_and_worst_element():
    want = torch.ones(3, 2, 4, dtype=torch.float64)
    got = want.clone()
    got[1, 0, 2] += 1e-3
    ok, ratio, steps, worst = R.check(got, want, want.abs(), 1e-5)
    assert not ok and ratio == pytest.approx(1e-3)
    assert steps[0] == 0 and steps[2] == 0 and steps[1] > 0
    assert worst == 1 * 8 + 0 * 4 + 2
    assert R.check(want.float(), want, want.abs(), 1e-5)[0]


def test_bump_is_one_bf16_ulp():
    t = torch.tensor([[1.0, -3.0], [0.25, 0.0]])
    s = torch.ones(2, 2, dtype=torch.float64)
    g = R.bump_one_ulp(t, t.double(), s)
    assert float(g[0, 1]) == -3.0 + 2.0 ** -6    # |-3| is the largest value against its scale: ulp(2..4) = 2^-6
    assert torch.equal(g.view(-1)[[0, 2, 3]], t.view(-1)[[0, 2, 3]])
    assert R.rne(torch.tensor([1.0 + 2.0 ** -8])).item() == 1.0                  # ties to even
    assert R.rne(torch.tensor([1.0 + 3 * 2.0 ** -8])).item() == 1.0 + 2.0 ** -6
