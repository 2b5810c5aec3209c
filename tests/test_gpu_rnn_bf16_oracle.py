"""The bf16 ReLU-RNN kernels checked step by step against the teacher-forced fp64 oracle (tests/rnn_bf16_oracle.py).

Entry points: tacorl_rnn_layer_fwd/bwd (PREC_BF16, one direction) and tacorl_rnn_layer2_fwd/bwd (a whole layer), over
the three recurrence engines behind them: per-step launches (gemm_tc_bf16), the 8-way persistent rnn_seq_kernel
("seq8") and the 4-CTA-cluster two-lane rnn_wave_kernel ("wave").  Every output is checked per element at
|got - want| <= TAU * S, S the same contraction on absolute values.

Calibration (NVIDIA B200, 1000 W power limit): TAU = 1e-5.  Largest |got - want| / S observed over every case of this
module: tacorl_rnn_layer_fwd 4.2e-7, tacorl_rnn_layer_bwd 6.1e-7, tacorl_rnn_layer2_fwd 4.9e-7, tacorl_rnn_layer2_bwd
5.8e-7, so TAU leaves 16x head room.  The discrimination controls fail by at least 20 * TAU = 2e-4 (asserted).

The engine a case takes is asserted, not assumed: the persistent kernels fall back to per-step launches silently.  The
same call at T + 8 steps adds at least 8 library launches on the per-step path and at most a few (a split-K decision
of a weight-gradient GEMM) on a persistent one.  seq8 performs exactly the per-step arithmetic, so a persistent run
bit-identical to the seq_enable = 0 run is seq8, and one that differs is the wave kernel (another K split)."""
import ctypes

import pytest
import torch

from tests import rnn_bf16_oracle as R
from tests.gpu_util import parity_report
from tests.rnn_bf16_oracle import TAU

pytestmark = pytest.mark.gpu

DEV = "cuda"
NAN = float("nan")
DT = 8                  # extra steps of the engine probe
WORST = {}              # entry point -> largest |err| / S seen
ENGINES = []            # (case, mode, fwd engine, bwd engine)


@pytest.fixture(scope="module")
def L():
    from tacorl_b200 import _lib
    lib = _lib.lib()
    was = lib.tacorl_rnn_seq_enable(1)
    yield _lib
    lib.tacorl_rnn_seq_enable(was)
    parity_report("rnn_bf16_oracle", [{"tau": TAU, "worst_err_over_scale": WORST,
                                       "engines": [list(e) for e in ENGINES]}])
    assert lib.tacorl_rnn_seq_timeouts() == 0      # (synchronises the device)


def _vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def _same(a, b):
    return torch.equal(_bits(a), _bits(b))


def _ws(nbytes):
    return torch.empty(int(nbytes), dtype=torch.uint8, device=DEV)


def _launches(L, fn):
    torch.cuda.synchronize()
    n0 = L.launch_count()
    fn()
    torch.cuda.synchronize()
    return L.launch_count() - n0


def _assert_ok(entry, tag, got, ref):
    """Every tensor of `got` within TAU * S of the oracle; records the worst ratio per entry point."""
    res = R.check_all(got, ref, TAU)
    for k, (ok, ratio, steps) in res.items():
        WORST[entry] = max(WORST.get(entry, 0.0), ratio)
        assert ok, f"{entry} {tag} {k}: max |err|/S = {ratio:.3e} > {TAU:g}; per-step rel L2 {[f'{s:.1e}' for s in steps]}"


def _rand_w(g, I, H):
    k = 1.0 / H ** 0.5
    return [((torch.rand(*s, generator=g) * 2 - 1) * k).to(DEV) for s in ((H, I), (H, H), (H,), (H,))]


def _engine(probe_delta, n):
    """Engine of a recurrence of n steps from the launch delta of the same call at n + DT steps."""
    if n <= 2:           # a chain of 0 or 1 steps is never persistent (rnn_seq_tc / rnn_wave_tc need >= 2)
        return "none" if n == 1 else "step"
    assert probe_delta >= DT or probe_delta <= DT // 2, f"launch delta {probe_delta} fits neither engine"
    return "step" if probe_delta >= DT else "persistent"


# ------------------------------------------------------------------------------------------ per-direction ABI
class Dir:
    """Inputs of one tacorl_rnn_layer_{fwd,bwd} case, laid out the way ReluRNNFn drives a bidirectional layer when
    `strided`: x a column slice of a wider buffer, out / dout at column offset d*H of a (T, B, 2H) buffer, lddx > I."""

    def __init__(self, T, B, I, H, reverse, n, h0, dhn, strided, acc, dxacc, seed):
        g = torch.Generator().manual_seed(seed)
        self.T, self.B, self.I, self.H, self.rev, self.n = T, B, I, H, int(reverse), n
        self.acc, self.dxacc = int(acc), int(dxacc)
        self.ldx = I + 16 if strided else I
        self.W = 2 * H if strided else H
        self.col = self.rev * H if strided else 0
        self.lddx = I + 8 if strided else I
        self.xbuf = torch.randn(T, B, self.ldx, generator=g).to(DEV)
        self.x = self.xbuf[..., :I]
        self.w_ih, self.w_hh, self.b_ih, self.b_hh = _rand_w(g, I, H)
        self.h0 = torch.rand(B, H, generator=g).to(DEV) if h0 else None
        self.dhn = torch.randn(B, H, generator=g).to(DEV) if dhn else None
        self.dout = torch.randn(T, B, H, generator=g).to(DEV)
        self.pre = {k: torch.randn(*s, generator=g).to(DEV) for k, s in
                    (("dw_ih", (H, I)), ("dw_hh", (H, H)), ("db_ih", (H,)), ("db_hh", (H,)), ("dx", (T, B, I)))}

    def fwd(self, L, tw_ih=None, tw_hh=None, T=None, n=None):
        T, n = T or self.T, n or self.n
        B, I, H = self.B, self.I, self.H
        x = self.x if T == self.T else torch.randn(T, B, I, device=DEV)
        obuf = torch.full((T, B, self.W), NAN, device=DEV)
        hb = torch.full((T, B, H), NAN, device=DEV, dtype=torch.bfloat16)
        ws = _ws(L.query("tacorl_rnn_layer_ws_bytes", T, B, I, H))
        k = _launches(L, lambda: L.call(
            "tacorl_rnn_layer_fwd", T, B, I, H, _vp(x), x.stride(1), _vp(self.w_ih), _vp(self.w_hh), _vp(self.b_ih),
            _vp(self.b_hh), _vp(self.h0), self.rev, n, _vp(obuf[..., self.col:]), self.W, _vp(tw_ih), _vp(tw_hh), _vp(hb),
            _vp(ws), ws.numel(), L.PREC_BF16, L.stream()))
        return {"obuf": obuf, "out": obuf[..., self.col:self.col + H], "hb": hb, "launches": k}

    def bwd(self, L, f, tw_ih=None, tw_hht=None, h_bf16=None, T=None, n=None):
        T, n = T or self.T, n or self.n
        B, I, H = self.B, self.I, self.H
        x = self.x if T == self.T else torch.randn(T, B, I, device=DEV)
        dbuf = torch.full((T, B, self.W), NAN, device=DEV)
        dbuf[..., self.col:self.col + H] = self.dout if T == self.T else torch.randn(T, B, H, device=DEV)
        dxbuf = torch.full((T, B, self.lddx), NAN, device=DEV)
        if self.dxacc and T == self.T:
            dxbuf[..., :I] = self.pre["dx"]
        g = {k: (self.pre[k].clone() if self.acc else torch.full_like(self.pre[k], NAN)) for k in ("dw_ih", "dw_hh", "db_ih", "db_hh")}
        g["dh0"] = torch.full((B, H), NAN, device=DEV)
        ws = _ws(L.query("tacorl_rnn_layer_ws_bytes", T, B, I, H))
        k = _launches(L, lambda: L.call(
            "tacorl_rnn_layer_bwd", T, B, I, H, _vp(x), x.stride(1), _vp(self.w_ih), _vp(self.w_hh), _vp(self.h0),
            self.rev, n, _vp(f["obuf"][..., self.col:]), self.W, _vp(dbuf[..., self.col:]), self.W, _vp(self.dhn),
            _vp(dxbuf), self.lddx, self.dxacc, _vp(g["dw_ih"]), _vp(g["dw_hh"]), _vp(g["db_ih"]), _vp(g["db_hh"]), self.acc,
            _vp(g["dh0"]), _vp(tw_ih), _vp(tw_hht), _vp(h_bf16), _vp(ws), ws.numel(), L.PREC_BF16, L.stream()))
        g.update(dbuf=dbuf, dpre=dbuf[..., self.col:self.col + H], dxbuf=dxbuf, dx=dxbuf[..., :I], launches=k)
        return g

    def check(self, L, f, b, tag):
        T, H, a = self.T, self.H, R.active(self.T, self.n, self.rev)
        out = f["out"]
        ref = R.fwd(self.x, self.w_ih, self.w_hh, self.b_ih, self.b_hh, out, self.h0, self.rev, self.n)
        _assert_ok("tacorl_rnn_layer_fwd", tag, {"out": out[a]}, ref)
        # the bf16 twin is the RNE of the fp32 state, written over the active steps only; nothing else is touched
        assert _same(f["hb"][a], out[a].bfloat16())
        act = torch.zeros(T, dtype=torch.bool, device=DEV)
        act[a] = True
        assert f["hb"][~act].isnan().all() and out[~act].isnan().all()
        other = torch.ones(self.W, dtype=torch.bool, device=DEV)
        other[self.col:self.col + H] = False
        assert f["obuf"][..., other].isnan().all() and b["dbuf"][..., other].isnan().all()
        ref = R.bwd(self.x, self.w_ih, self.w_hh, out, self.dout, b["dpre"], self.h0, self.dhn, self.rev, self.n)
        got = {"dpre": b["dpre"][a], "dx": b["dx"][a], "dh0": b["dh0"]}
        if self.dxacc:
            ref["dx"] = (ref["dx"][0] + self.pre["dx"][a].double(), ref["dx"][1] + self.pre["dx"][a].double().abs())
        for k, r in (("dw_ih", "dw_ih"), ("dw_hh", "dw_hh"), ("db_ih", "db"), ("db_hh", "db")):
            want, s = ref[r]
            ref[k] = (want + self.pre[k].double(), s + self.pre[k].double().abs()) if self.acc else (want, s)
            got[k] = b[k]
        del ref["db"]
        _assert_ok("tacorl_rnn_layer_bwd", tag, got, ref)
        assert torch.equal(b["dpre"][~act], self.dout[~act])          # steps outside the recurrence keep dL/dout
        want_dx = self.pre["dx"][~act] if self.dxacc else torch.zeros_like(b["dx"][~act])
        assert _same(b["dx"][~act], want_dx)                           # zeroed rows (or the accumulated ones)
        assert b["dxbuf"][..., self.I:].isnan().all()
        if not self.acc:
            assert _same(b["db_ih"], b["db_hh"])


# (T, B, I, H, reverse, n, h0, dhn, strided, accumulate, dx_accumulate, engine with seq_enable = 1)
DIR_CASES = [
    (16, 64, 48, 2048, 0, 16, 1, 1, 0, 0, 0, "seq8"),
    (16, 64, 48, 2048, 1, 13, 1, 1, 1, 1, 0, "seq8"),
    (16, 128, 2048, 2048, 0, 16, 0, 0, 1, 0, 1, "seq8"),     # M = 128: the 8-way kernel's limit
    (16, 128, 2048, 2048, 1, 1, 1, 1, 0, 1, 0, "none"),
    (9, 129, 64, 1024, 0, 9, 1, 1, 1, 0, 0, "step"),         # B > 128: per-step even when enabled
    (9, 129, 64, 1024, 1, 6, 0, 1, 0, 1, 1, "step"),
    (5, 3, 12, 256, 1, 5, 1, 1, 1, 1, 1, "step"),            # I % 8 != 0, H = 256 (K % 512 != 0): per-step
    (5, 3, 12, 256, 0, 2, 1, 0, 0, 0, 0, "step"),
    (7, 24, 33, 512, 0, 4, 1, 1, 1, 0, 1, "seq8"),
    (7, 24, 33, 512, 1, 7, 0, 0, 0, 1, 0, "seq8"),
    (1, 64, 48, 2048, 0, 1, 1, 1, 0, 0, 0, "none"),          # T = 1
    (1, 24, 33, 512, 1, 1, 0, 1, 1, 0, 1, "none"),
]


@pytest.mark.parametrize("mode", [1, 0])
@pytest.mark.parametrize("case", DIR_CASES, ids=lambda c: "T{}B{}I{}H{}r{}n{}h0{}dhn{}s{}a{}{}".format(*c[:11]))
def test_rnn_layer_bf16_matches_teacher_forced_oracle(L, case, mode):
    T, B, I, H, rev, n, h0, dhn, strided, acc, dxacc, engine = case
    L.lib().tacorl_rnn_seq_enable(mode)
    try:
        c = Dir(T, B, I, H, rev, n, h0, dhn, strided, acc, dxacc, seed=T * 1000 + B * 7 + I + H + rev + n)
        f = c.fwd(L)
        b = c.bwd(L, f)
        c.check(L, f, b, f"mode {mode}")
        if n >= 3:
            pf = c.fwd(L, T=T + DT, n=n + DT)
            pb = c.bwd(L, pf, T=T + DT, n=n + DT)
            got = (_engine(pf["launches"] - f["launches"], n), _engine(pb["launches"] - b["launches"], n))
        else:
            got = (_engine(0, n),) * 2
    finally:
        L.lib().tacorl_rnn_seq_enable(1)
    got = tuple("seq8" if e == "persistent" else e for e in got)    # the only persistent engine of these entry points
    want = "step" if (mode == 0 and engine != "none") else engine
    ENGINES.append(("layer T{} B{} I{} H{} rev{} n{}".format(T, B, I, H, rev, n), mode, *got))
    assert got == (want, want), (got, want)


@pytest.mark.parametrize("case", [DIR_CASES[0], DIR_CASES[1], DIR_CASES[6], DIR_CASES[9]],
                         ids=lambda c: "T{}B{}I{}H{}r{}n{}".format(*c[:6]))
def test_rnn_layer_bf16_twins_bit_identical_to_staging(L, case):
    """Caller-supplied bf16 twins (w_ih_bf16, w_hh_bf16, W_hh^T from tacorl_cast_transpose_bf16, the forward's own
    h_bf16_out) give bit-identical results to the staged casts, and twins that are not 16-byte aligned (offset by 2
    bytes) fall back to staging."""
    T, B, I, H, rev, n, h0, dhn, strided, acc, dxacc, _ = case
    c = Dir(T, B, I, H, rev, n, h0, dhn, strided, acc, dxacc, seed=99 + T + B)
    wt = torch.empty(H, H, device=DEV, dtype=torch.bfloat16)
    L.call("tacorl_cast_transpose_bf16", _vp(c.w_hh), H, H, _vp(wt), L.stream())
    assert _same(wt, c.w_hh.bfloat16().t())
    twins = [c.w_ih.bfloat16(), c.w_hh.bfloat16(), wt]

    def shifted(t):       # same values, 2 bytes off a 16-byte boundary
        buf = torch.empty(t.numel() + 1, device=DEV, dtype=torch.bfloat16)
        buf[1:] = t.reshape(-1)
        return buf[1:]

    f0 = c.fwd(L)
    b0 = c.bwd(L, f0)
    for tw in (twins, [shifted(t) for t in twins]):
        f = c.fwd(L, tw[0], tw[1])
        assert _same(f["obuf"], f0["obuf"]) and _same(f["hb"], f0["hb"])
        b = c.bwd(L, f0, tw[0], tw[2], f0["hb"] if tw is twins else shifted(f0["hb"]))
        for k in ("dbuf", "dxbuf", "dw_ih", "dw_hh", "db_ih", "db_hh", "dh0"):
            assert _same(b[k], b0[k]), k


# ------------------------------------------------------------------------------------------ whole-layer ABI
class Layer2:
    """Inputs of one tacorl_rnn_layer2_{fwd,bwd} case: (T, B, D*H) outputs, bf16 twins in the same layout."""

    def __init__(self, T, B, I, H, D, n1, grad_rows, xb, seed):
        g = torch.Generator().manual_seed(seed)
        self.T, self.B, self.I, self.H, self.D, self.Bg = T, B, I, H, D, grad_rows or B
        self.nst = [T] + ([n1] if D == 2 else [])
        self.gr = grad_rows
        self.x = torch.randn(T, B, I, generator=g).to(DEV)
        self.xb = self.x.bfloat16() if xb else None
        self.w = [w for _ in range(D) for w in _rand_w(g, I, H)]
        self.dout = torch.randn(T, B, D * H, generator=g).to(DEV)
        self.dout[:, self.Bg:] = 0            # rows behind grad_rows carry no gradient

    def fwd(self, L, T=None, nst=None):
        T, nst = T or self.T, nst or self.nst
        B, I, H, D = self.B, self.I, self.H, self.D
        x = self.x if T == self.T else torch.randn(T, B, I, device=DEV)
        xb = None if self.xb is None else x.bfloat16()
        out = torch.full((T, B, D * H), NAN, device=DEV)
        outb = torch.full((T, B, D * H), NAN, device=DEV, dtype=torch.bfloat16)
        ws = _ws(L.query("tacorl_rnn_layer2_ws_bytes", T, B, I, H, D))
        k = _launches(L, lambda: L.call(
            "tacorl_rnn_layer2_fwd", T, B, I, H, D, _vp(x), I, _vp(xb), I, L.ptr_array(self.w), None, L.int_array(nst),
            _vp(out), D * H, _vp(outb), _vp(ws), ws.numel(), L.stream()))
        return {"out": out, "outb": outb, "launches": k}

    def bwd(self, L, f, T=None, nst=None):
        T, nst = T or self.T, nst or self.nst
        B, I, H, D = self.B, self.I, self.H, self.D
        x = self.x if T == self.T else torch.randn(T, B, I, device=DEV)
        xb = None if self.xb is None else x.bfloat16()
        dbuf = self.dout.clone() if T == self.T else torch.zeros(T, B, D * H, device=DEV)
        # rows behind grad_rows must read as zeros; otherwise every element BPTT writes starts as a NaN sentinel
        dpb = torch.full((T, B, D * H), 0.0 if self.Bg < B else NAN, device=DEV, dtype=torch.bfloat16)
        dx = torch.full((T, B, I), NAN, device=DEV)
        dw = [torch.full_like(w, NAN) for w in self.w]
        w2 = [self.w[4 * d + j] for d in range(D) for j in (0, 1)]
        ws = _ws(L.query("tacorl_rnn_layer2_ws_bytes", T, B, I, H, D))
        k = _launches(L, lambda: L.call(
            "tacorl_rnn_layer2_bwd", T, B, self.gr, I, H, D, _vp(x), I, _vp(xb), I, L.ptr_array(w2), None,
            L.int_array(nst), _vp(f["out"]), D * H, _vp(f["outb"]), _vp(dbuf), D * H, _vp(dpb), _vp(dx), I,
            L.ptr_array(dw), _vp(ws), ws.numel(), L.stream()))
        return {"dpre": dbuf, "dpb": dpb, "dx": dx, "dw": dw, "launches": k}

    def check_fwd(self, f, tag):
        T, H = self.T, self.H
        for d in range(self.D):
            n, cs = self.nst[d], slice(d * H, (d + 1) * H)
            a = R.active(T, n, d == 1)
            out = f["out"][..., cs]
            w_ih, w_hh, b_ih, b_hh = self.w[4 * d:4 * d + 4]
            ref = R.fwd(self.x, w_ih, w_hh, b_ih, b_hh, out, None, d == 1, n)
            _assert_ok("tacorl_rnn_layer2_fwd", f"{tag} d{d}", {"out": out[a]}, ref)
            assert _same(f["outb"][a, :, cs], out[a].bfloat16())
            if n < T:       # steps outside a direction's recurrence are not written
                rest = torch.ones(T, dtype=torch.bool, device=DEV)
                rest[a] = False
                assert f["out"][rest, :, cs].isnan().all() and f["outb"][rest, :, cs].isnan().all()

    def check_bwd(self, f, b, tag):
        """f: the forward whose outputs the backward call consumed."""
        T, B, H, D, Bg = self.T, self.B, self.H, self.D, self.Bg
        dx_ref = None
        for d in range(D):
            n, cs = self.nst[d], slice(d * H, (d + 1) * H)
            a = R.active(T, n, d == 1)
            out = f["out"][..., cs]
            w_ih, w_hh = self.w[4 * d:4 * d + 2]
            ref = R.bwd(self.x, w_ih, w_hh, out, self.dout[..., cs], b["dpre"][..., cs], None, None, d == 1, n)
            dpre = b["dpre"][a, :, cs]
            got = {"dpre": dpre, "dw_ih": b["dw"][4 * d], "dw_hh": b["dw"][4 * d + 1], "db_ih": b["dw"][4 * d + 2],
                   "db_hh": b["dw"][4 * d + 3]}
            ref["db_ih"] = ref["db_hh"] = ref.pop("db")
            dxd = ref.pop("dx")
            del ref["dh0"]
            _assert_ok("tacorl_rnn_layer2_bwd", f"{tag} d{d}", got, ref)
            # the bf16 twin of dpre: RNE of the fp32 value on the rows that carry a gradient, zero behind them
            assert _same(b["dpb"][a, :Bg, cs], dpre[:, :Bg].bfloat16())
            assert not b["dpb"][a, Bg:, cs].float().any() and not dpre[:, Bg:].any()
            full = [torch.zeros(T, B, self.I, dtype=torch.float64, device=DEV) for _ in range(2)]
            full[0][a], full[1][a] = dxd
            dx_ref = full if dx_ref is None else [dx_ref[0] + full[0], dx_ref[1] + full[1]]
            if n < T:       # steps outside a direction's recurrence keep dL/dout
                rest = torch.ones(T, dtype=torch.bool, device=DEV)
                rest[a] = False
                assert torch.equal(b["dpre"][rest, :, cs], self.dout[rest, :, cs])
        _assert_ok("tacorl_rnn_layer2_bwd", f"{tag} dx", {"dx": b["dx"]}, {"dx": tuple(dx_ref)})
        assert not b["dx"][:, Bg:].any()


# (T, B, I, H, D, n_steps[1], grad_rows, x_bf16 given, fwd engine, bwd engine with seq_enable = 1)
L2_CASES = [
    (16, 64, 48, 2048, 2, 1, 0, 1, "wave", "wave"),          # the BiRNN's last_only top layer
    (16, 64, 2048, 1024, 2, 1, 16, 1, "wave", "wave"),       # reverse input projection: M = 64, cluster split-K
    (16, 63, 12, 1024, 1, 0, 0, 0, "wave", "wave"),
    (5, 24, 48, 512, 2, 5, 1, 1, "wave", "wave"),
    (5, 3, 12, 256, 2, 5, 0, 0, "wave", "wave"),             # 3 rows: the wave kernel's per-rank rows half empty
    (16, 3, 512, 256, 1, 0, 0, 1, "wave", "wave"),
    (16, 64, 512, 256, 2, 16, 63, 0, "wave", "wave"),
    (5, 64, 12, 1024, 1, 0, 1, 0, "wave", "wave"),
    (16, 65, 48, 1024, 1, 0, 0, 1, "seq8", "seq8"),
    (16, 128, 48, 2048, 1, 0, 0, 1, "seq8", "seq8"),
    (16, 128, 4096, 2048, 1, 0, 63, 1, "seq8", "wave"),      # BPTT over 63 rows: back in the wave kernel
    (16, 128, 48, 2048, 2, 1, 16, 1, "step", "wave"),
    (16, 100, 2048, 1024, 2, 16, 0, 1, "step", "step"),
    (5, 200, 48, 512, 1, 0, 0, 1, "step", "step"),
    (2, 64, 1024, 512, 2, 2, 0, 1, "step", "step"),          # T*B = 128: both input projections cluster split-K
    (1, 100, 1024, 512, 2, 1, 0, 1, "none", "none"),         # T = 1: a single step, cluster split-K
]


@pytest.mark.parametrize("case", L2_CASES, ids=lambda c: "T{}B{}I{}H{}D{}n{}g{}xb{}".format(*c[:8]))
def test_rnn_layer2_bf16_matches_teacher_forced_oracle(L, case):
    """seq_enable 1, 0 and (two directions) 2: every run checked against the oracle; mode 2 launches the two lanes one
    after the other and must be bit-identical to mode 1."""
    T, B, I, H, D, n1, gr, xb, e_fwd, e_bwd = case
    lib = L.lib()
    c = Layer2(T, B, I, H, D, n1, gr, xb, seed=T * 1000 + B * 7 + I + H + D + n1 + gr)
    runs = {}
    try:
        for mode in ([1, 0, 2] if D == 2 else [1, 0]):
            lib.tacorl_rnn_seq_enable(mode)
            f = c.fwd(L)
            c.check_fwd(f, f"mode {mode}")
            f1 = runs[1][0] if mode != 1 else f    # BPTT of every mode on the same forward: comparable bit for bit
            runs[mode] = (f, c.bwd(L, f1))
            c.check_bwd(f1, runs[mode][1], f"mode {mode}")
        lib.tacorl_rnn_seq_enable(1)
        n = T           # (the longest chain of the layer: the forward direction's)
        nst = [v + DT if v > 1 else v for v in c.nst]
        if n >= 3:
            pf = c.fwd(L, T + DT, nst)
            pb = c.bwd(L, pf, T + DT, nst)
            got = [_engine(pf["launches"] - runs[1][0]["launches"], n), _engine(pb["launches"] - runs[1][1]["launches"], n)]
        else:
            got = [_engine(0, n)] * 2
    finally:
        lib.tacorl_rnn_seq_enable(1)
    f1, b1 = runs[1]
    f0, b0 = runs[0]
    if got[0] == "persistent":
        got[0] = "seq8" if _same(f1["out"], f0["out"]) else "wave"
    if got[1] == "persistent":
        got[1] = "seq8" if _same(b1["dpre"], b0["dpre"]) else "wave"
    ENGINES.append(("layer2 T{} B{} I{} H{} D{} n{} g{}".format(T, B, I, H, D, n1, gr), 1, *got))
    assert tuple(got) == (e_fwd, e_bwd), (got, (e_fwd, e_bwd))
    if D == 2:
        f2, b2 = runs[2]
        for k in ("out", "outb"):
            assert _same(f2[k], f1[k]), k
        for k in ("dpre", "dpb", "dx"):
            assert _same(b2[k], b1[k]), k
        assert all(_same(u, v) for u, v in zip(b2["dw"], b1["dw"]))
        if e_fwd == "wave" and n1 > 2:   # two lanes: one launch more when launched one after the other
            assert f2["launches"] == f1["launches"] + 1


# ------------------------------------------------------------------------------------------ discrimination controls
def test_oracle_check_catches_subtle_errors_on_kernel_data(L):
    """On one kernel run with h0 and dhn: the check of the unaltered oracle passes, and each control (an oracle altered
    the way a subtle kernel bug would be, or a copy of one kernel output moved by one bf16 ulp) fails it by at least
    20x TAU."""
    c = Dir(16, 64, 48, 2048, 1, 13, 1, 1, 1, 0, 0, seed=4242)
    f = c.fwd(L)
    b = c.bwd(L, f)
    a = R.active(c.T, c.n, True)
    got = {"out": f["out"][a], "dpre": b["dpre"][a], "dw_ih": b["dw_ih"], "dw_hh": b["dw_hh"], "db": b["db_ih"],
           "dx": b["dx"][a], "dh0": b["dh0"]}

    def oracle(control=None):
        ref = R.fwd(c.x, c.w_ih, c.w_hh, c.b_ih, c.b_hh, f["out"], c.h0, True, c.n, control)
        ref.update(R.bwd(c.x, c.w_ih, c.w_hh, f["out"], c.dout, b["dpre"], c.h0, c.dhn, True, c.n, control))
        return ref

    ref = oracle()
    assert all(r[0] for r in R.check_all(got, ref, TAU).values())
    for control in R.CONTROLS:
        res = R.check_all(got, oracle(control), TAU)
        worst = max(r[1] for r in res.values())
        assert worst >= 20 * TAU, (control, {k: r[1] for k, r in res.items()})
    for k in got:
        ok, ratio, _, _ = R.check(R.bump_one_ulp(got[k], *ref[k]), *ref[k], TAU)
        assert not ok and ratio >= 20 * TAU, (k, ratio)


# ------------------------------------------------------------------------------------------ model-level bridge
@pytest.fixture
def bf16_ops(L):
    from tacorl_b200 import ops
    ops.set_precision("bf16")
    yield ops
    ops.set_precision("fp32")


def test_relu_rnn2_bidirectional_last_only_is_the_verified_abi_chain(L, bf16_ops):
    """ops.relu_rnn (ReluRNN2Fn: 2 layers, bidirectional, last_only) equals, bit for bit in the output and every
    gradient, the chain of tacorl_rnn_layer2 calls the tests above verify."""
    T, B, I, H, D = 16, 64, 48, 1024, 2
    g = torch.Generator().manual_seed(7)
    w = [t for l in range(2) for _ in range(D) for t in _rand_w(g, I if l == 0 else D * H, H)]
    x = torch.randn(T, B, I, generator=g).to(DEV)
    cot = torch.randn(B, D * H, generator=g).to(DEV)
    ws = [t.clone().requires_grad_(True) for t in w]
    xd = x.clone().requires_grad_(True)
    y, _ = bf16_ops.relu_rnn(xd, ws, 2, True, True)
    (y * cot).sum().backward()
    torch.cuda.synchronize()
    # the same work through the ABI
    outs, inp, inp_b = [], x, None
    for l in range(2):
        Il = inp.shape[2]
        out = torch.empty(T, B, D * H, device=DEV)
        outb = torch.empty(T, B, D * H, device=DEV, dtype=torch.bfloat16)
        nst = [T, 1 if l == 1 else T]
        buf = _ws(L.query("tacorl_rnn_layer2_ws_bytes", T, B, Il, H, D))
        L.call("tacorl_rnn_layer2_fwd", T, B, Il, H, D, _vp(inp), Il, _vp(inp_b), Il, L.ptr_array(w[8 * l:8 * l + 8]), None,
               L.int_array(nst), _vp(out), D * H, _vp(outb), _vp(buf), buf.numel(), L.stream())
        outs.append((inp, inp_b, out, outb, nst))
        inp, inp_b = out, outb
    assert _same(y, inp[T - 1])
    dbuf = torch.zeros(T, B, D * H, device=DEV)
    dbuf[T - 1] = cot
    grads = [None] * len(w)
    for l in (1, 0):
        inp, inp_b, out, outb, nst = outs[l]
        Il = inp.shape[2]
        wl = w[8 * l:8 * l + 8]
        w2 = [wl[4 * d + j] for d in range(D) for j in (0, 1)]
        dpb = torch.empty(T, B, D * H, device=DEV, dtype=torch.bfloat16)
        dx = torch.empty(T, B, Il, device=DEV)
        dw = [torch.empty_like(t) for t in wl]
        buf = _ws(L.query("tacorl_rnn_layer2_ws_bytes", T, B, Il, H, D))
        L.call("tacorl_rnn_layer2_bwd", T, B, 0, Il, H, D, _vp(inp), Il, _vp(inp_b), Il, L.ptr_array(w2), None,
               L.int_array(nst), _vp(out), D * H, _vp(outb), _vp(dbuf), D * H, _vp(dpb), _vp(dx), Il, L.ptr_array(dw),
               _vp(buf), buf.numel(), L.stream())
        grads[8 * l:8 * l + 8] = dw
        dbuf = dx
    torch.cuda.synchronize()
    assert _same(xd.grad, dbuf)
    for i, (p, want) in enumerate(zip(ws, grads)):
        assert _same(p.grad, want), i


def test_relu_rnn_with_h0_is_the_verified_abi_chain(L, bf16_ops):
    """ops.relu_rnn with a carried hidden state (ReluRNNFn, the rollout path: 1 layer, h0) equals, bit for bit in the
    output, h_n and every gradient (dh0 included), the per-direction ABI calls the tests above verify."""
    T, B, I, H = 16, 64, 48, 2048
    g = torch.Generator().manual_seed(11)
    w = _rand_w(g, I, H)
    x = torch.randn(T, B, I, generator=g).to(DEV)
    h0 = torch.rand(1, B, H, generator=g).to(DEV)
    cot, cot_h = torch.randn(T, B, H, generator=g).to(DEV), torch.randn(1, B, H, generator=g).to(DEV)
    ws = [t.clone().requires_grad_(True) for t in w]
    xd, h0d = x.clone().requires_grad_(True), h0.clone().requires_grad_(True)
    y, hn = bf16_ops.relu_rnn(xd, ws, 1, False, False, h0d)
    ((y * cot).sum() + (hn * cot_h).sum()).backward()
    torch.cuda.synchronize()
    out = torch.empty(T, B, H, device=DEV)
    hb = torch.empty(T, B, H, device=DEV, dtype=torch.bfloat16)
    buf = _ws(L.query("tacorl_rnn_layer_ws_bytes", T, B, I, H))
    L.call("tacorl_rnn_layer_fwd", T, B, I, H, _vp(x), I, *[_vp(t) for t in w], _vp(h0[0]), 0, T, _vp(out), H, None, None,
           _vp(hb), _vp(buf), buf.numel(), L.PREC_BF16, L.stream())
    assert _same(y, out) and _same(hn[0], out[T - 1])
    wt = torch.empty(H, H, device=DEV, dtype=torch.bfloat16)
    L.call("tacorl_cast_transpose_bf16", _vp(w[1]), H, H, _vp(wt), L.stream())
    dbuf = cot.clone()
    dx, dh0 = torch.empty(T, B, I, device=DEV), torch.empty(B, H, device=DEV)
    dw = [torch.empty_like(t) for t in w]
    L.call("tacorl_rnn_layer_bwd", T, B, I, H, _vp(x), I, _vp(w[0]), _vp(w[1]), _vp(h0[0]), 0, T, _vp(out), H, _vp(dbuf), H,
           _vp(cot_h[0]), _vp(dx), I, 0, *[_vp(t) for t in dw], 0, _vp(dh0), None, _vp(wt), _vp(hb), _vp(buf), buf.numel(),
           L.PREC_BF16, L.stream())
    torch.cuda.synchronize()
    assert _same(xd.grad, dx) and _same(h0d.grad[0], dh0)
    for i, (p, want) in enumerate(zip(ws, dw)):
        assert _same(p.grad, want), i
