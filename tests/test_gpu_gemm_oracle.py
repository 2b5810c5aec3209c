"""Every route and epilogue of the GEMM family checked per element against the fp64 oracle (tests/gemm_oracle.py),
with the route each case takes asserted.

The bf16 tensor-core kernels run through tacorl_gemm_tc_debug, which reports the kernel that ran (tiled or skinny
cluster, BN or NT, z-slices, CTAs); each row of gemm_oracle.GEMM_CASES names that route for each operand layout and the
test asserts it.  Operands are bf16-exact and sit in buffers whose padded pitch holds NaN, which the tensor maps must
never read.  Outputs (C, Cb, Cpre) are windows of NaN-filled wider buffers, at a base offset and pitch that pick the
vector epilogue ("vec") or the scalar one ("scalar"); the gate is a window of its own with 0.0, -0.0 and negatives.  On
every route, for every epilogue of gemm_oracle.EPILOGUES:
  - C, Cpre within TAU * S of the oracle and Cb within that plus half a bf16 ulp, per element;
  - Cb equal to the bf16 round-to-nearest of the kernel's own C, bit for bit; with ReLU, C equal to the gated
    relu(Cpre); gated elements exactly +0;
  - every element outside [M, N] of every output still NaN; with beta == 0 the NaN-filled C never leaks in.
On the full epilogue ("all") of every route: a second run and a run with a zero-filled instead of a 0xFF-filled (NaN)
workspace are bit-identical (every split-K partial slice is written before it is read), and every control of the
oracle, and a one-ulp bump of one Cb element, fails the check by at least 20 * TAU.

ops.gemm at bf16 precision: below 2^24 multiply-adds the fp32 SIMT kernels run (launch count, and a result that holds
TAU on the unrounded operands where the bf16-rounded ones miss it); bf16 shadow operands give results bit-identical to
staged ones with one cast launch fewer each; a shadow whose pitch is not a multiple of 8 is ignored (a NaN shadow
changes nothing).  ops.gemm at fp32 precision: all four transpose combinations on each sgemm tile shape and the
automatic split-K with SiLU and Cpre, launch counts asserted.

Calibration, measured on an NVIDIA B200 at its 1000 W power limit (the parity report "gemm_oracle" lists, per case,
the worst |err| / S and, per control, its ratio to TAU): the worst |err| / S over all cases is 8.3e-7 = TAU / 12 (the
tiled kernel at K = 8192 on the skinny fallback; tiled 3.1e-7, split-K 9.2e-8, skinny cluster 4.6e-7, sgemm 3.3e-7).
The weakest control is the one-ulp Cb bump at 53 TAU; drop_last_kblock fails by at least 520 TAU, act_before_bias by
5800 TAU, the others by 9700 TAU or more."""
import ctypes

import pytest
import torch

from tests import gemm_oracle as G
from tests.gemm_oracle import TAU
from tests.gpu_util import parity_report

pytestmark = pytest.mark.gpu

DEV = "cuda"
NAN = float("nan")
WORST = {}            # case -> {output: largest |err| / S over its epilogues and placements}
CONTROLS = {}         # case -> {control: largest ratio over the outputs / TAU}
ROUTES = {}           # case -> route reported by the library


@pytest.fixture(scope="module")
def L():
    from tacorl_b200 import _lib
    _lib.lib()
    yield _lib
    parity_report("gemm_oracle", [{"tau": TAU, "worst_err_over_scale": WORST, "controls_over_tau": CONTROLS,
                                   "routes": ROUTES}])


def _vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def _pad8(n):
    return (n + 7) // 8 * 8


def _launches(L, fn):
    torch.cuda.synchronize()
    n0 = L.launch_count()
    fn()
    torch.cuda.synchronize()
    return L.launch_count() - n0


def stored_bf16(t):
    """t (bf16-exact) on the device as bf16 with its pitch padded to a multiple of 8 elements; the padding is NaN."""
    r, c = t.shape
    buf = torch.full((r, _pad8(c)), NAN, dtype=torch.bfloat16, device=DEV)
    buf[:, :c] = t.to(DEV).bfloat16()
    return buf


class Window:
    """An M x N window of a NaN-filled (M + 2) x ld buffer, from row 1.  "vec": column 0 and ld a multiple of 8 (16-byte
    aligned rows); "scalar": column 1 and an odd ld."""

    def __init__(self, M, N, dtype, place, init=None):
        self.ld = _pad8(N) + 8 + (1 if place == "scalar" else 0)
        self.off = 1 if place == "scalar" else 0
        self.buf = torch.full((M + 2, self.ld), NAN, dtype=dtype, device=DEV)
        self.view = self.buf[1:M + 1, self.off:self.off + N]
        if init is not None:
            self.view.copy_(init)

    def outside_is_nan(self):
        keep = torch.ones(self.buf.shape, dtype=torch.bool, device=DEV)
        keep[1:self.view.shape[0] + 1, self.off:self.off + self.view.shape[1]] = False
        return bool(self.buf[keep].isnan().all())


class Case:
    """Operands and epilogue inputs of one (row, layout) of gemm_oracle.GEMM_CASES, with the fp64 products."""

    def __init__(self, name, layout):
        self.name, self.layout = name, layout
        self.M, self.N, self.K, self.split_k, self.ws_bytes, self.places, routes = G.GEMM_CASES[name]
        self.route = routes[layout]
        self.a_mn, self.b_mn = G.LAYOUTS[layout]
        M, N, K = self.M, self.N, self.K
        g = torch.Generator().manual_seed(M * 131 + N * 7 + K + 1000 * self.a_mn + 2000 * self.b_mn)
        A, B = G.make_operands(g, M, N, K, self.a_mn, self.b_mn)
        C0, bias, gate = G.make_epilogue_inputs(g, M, N, K)
        self.A, self.B = stored_bf16(A), stored_bf16(B)
        self.C0, self.gate = C0.to(DEV), gate.to(DEV)
        self.bias = bias.to(DEV)
        self.bias_off = torch.full((N + 1,), NAN, device=DEV)     # the same bias one element off 16-byte alignment
        self.bias_off[1:] = self.bias
        self.P = G.Products(G.op_a(A.to(DEV), self.a_mn), G.op_b(B.to(DEV), self.b_mn))

    def fields(self, ep):
        return dict(alpha=ep.get("alpha", 1.0), beta=ep.get("beta", 0.0), C0=self.C0 if ep.get("beta") else None,
                    bias=self.bias if ep.get("bias") else None, act=ep.get("act", G.ACT_NONE),
                    gate=self.gate if ep.get("gate") else None)

    def run(self, L, ep, place, ws_fill=0xFF):
        M, N = self.M, self.N
        f = self.fields(ep)
        C = Window(M, N, torch.float32, place, self.C0 if f["beta"] else None) if ep.get("c") else None
        Cb = Window(M, N, torch.bfloat16, place) if ep.get("cb") else None
        Cpre = Window(M, N, torch.float32, place) if ep.get("cpre") else None
        gate = Window(M, N, torch.float32, place, self.gate) if ep.get("gate") else None
        bias = (self.bias if place == "vec" else self.bias_off[1:]) if ep.get("bias") else None
        ws = torch.full((self.ws_bytes,), ws_fill, dtype=torch.uint8, device=DEV) if self.ws_bytes else None
        route = (ctypes.c_int * 4)()
        torch.cuda.synchronize()
        L.call("tacorl_gemm_tc_debug", _vp(self.A), self.A.stride(0), self.a_mn, _vp(self.B), self.B.stride(0),
               self.b_mn, M, N, self.K, float(f["alpha"]), float(f["beta"]), _vp(C and C.view), C.ld if C else 0,
               _vp(Cb and Cb.view), Cb.ld if Cb else 0, _vp(bias), int(f["act"]), _vp(Cpre and Cpre.view),
               Cpre.ld if Cpre else 0, self.split_k, _vp(gate and gate.view), gate.ld if gate else 0, _vp(ws),
               self.ws_bytes or 0, ctypes.c_void_p(ctypes.addressof(route)), L.stream())
        torch.cuda.synchronize()
        return {"out": C, "cb": Cb, "pre": Cpre, "route": tuple(route)}


def _check_outputs(case, o, ep, f, tag, worst):
    ref = G.reference(case.P, **f)
    for k, r in ref.items():
        if o[k] is None:
            continue
        ok, ratio, idx = G.check(o[k].view, *r[:2], TAU, bf16=len(r) > 2)
        worst[k] = max(worst.get(k, 0.0), ratio)
        assert ok, (tag, k, ratio, idx)
        assert o[k].outside_is_nan(), (tag, k, "wrote outside [M, N]")
    C, Cb, Cpre = o["out"], o["cb"], o["pre"]
    if C is not None and Cb is not None:
        assert torch.equal(_bits(Cb.view), _bits(C.view.bfloat16())), (tag, "Cb is not rne(C)")
    gated = (case.gate <= 0) if f["gate"] is not None else None
    if C is not None and Cpre is not None and f["act"] == G.ACT_RELU:
        want = torch.relu(Cpre.view)
        if gated is not None:
            want = torch.where(gated, torch.zeros_like(want), want)
        assert torch.equal(C.view, want), (tag, "C is not relu(Cpre)")
    if gated is not None:
        for w in (C, Cb):
            if w is not None:
                assert bool((_bits(w.view)[gated] == 0).all()), (tag, "a gated element is not +0")
    return ref


CASES = [(n, lay) for n, c in G.GEMM_CASES.items() for lay in c[6]]


@pytest.mark.parametrize("name,layout", CASES)
def test_gemm_tc_route_epilogues_and_controls(L, name, layout):
    case = Case(name, layout)
    tag0 = f"{name}/{layout}"
    worst, ctl = {}, {}
    for place in case.places:
        for en, ep in G.EPILOGUES.items():
            tag = f"{tag0}/{place}/{en}"
            f = case.fields(ep)
            o = case.run(L, ep, place)
            assert o["route"] == case.route, (tag, o["route"], case.route)
            ref = _check_outputs(case, o, ep, f, tag, worst)
            if en != "all" or place != case.places[0]:
                continue
            for ws_fill in (0xFF, 0x00):          # a second run; a workspace of zeros instead of NaN
                o2 = case.run(L, ep, place, ws_fill)
                for k in ("out", "cb", "pre"):
                    if o[k] is not None:
                        assert torch.equal(_bits(o2[k].buf), _bits(o[k].buf)), (tag, k, "run to run", ws_fill)
            for control in G.CONTROLS:
                bad = G.reference(case.P, control=control, **f)
                r = max(G.check(o[k].view, *bad[k][:2], TAU, bf16=len(bad[k]) > 2)[1] for k in bad)
                ctl[control] = r / TAU
                assert r >= 20 * TAU, (tag, control, r)
            want, scale = ref["cb"][:2]
            ok, r, _ = G.check(G.bump_one_ulp(o["cb"].view.contiguous(), want, scale), want, scale, TAU, bf16=True)
            ctl["cb_one_ulp"] = r / TAU
            assert not ok and r >= 20 * TAU, (tag, "cb_one_ulp", r)
    WORST[tag0], CONTROLS[tag0], ROUTES[tag0] = worst, ctl, list(case.route)


# ------------------------------------------------------------------------------------------ through ops.gemm
@pytest.fixture
def ops_bf16():
    from tacorl_b200 import ops
    ops.set_precision("bf16")
    yield ops
    ops.set_precision("fp32")


def _ops_case(g, M, N, K, tA, tB, exact):
    A = torch.randn((K, M) if tA else (M, K), generator=g)
    B = torch.randn((N, K) if tB else (K, N), generator=g)
    if exact:
        A, B = A.bfloat16().float(), B.bfloat16().float()
    C0, bias, _ = G.make_epilogue_inputs(g, M, N, K)
    return A.to(DEV), B.to(DEV), C0.to(DEV), bias.to(DEV)


def _products(A, B, tA, tB, rounded=False):
    a, b = (G.rne(A), G.rne(B)) if rounded else (A.double(), B.double())
    return G.Products(a.t() if tA else a, b.t() if tB else b)


def test_ops_bf16_below_2pow24_runs_the_fp32_kernels(L, ops_bf16):
    M, N, K = 64, 64, 1000
    assert G.ops_bf16_route(M, N, K) == "f32"
    g = torch.Generator().manual_seed(5)
    A, B, C0, bias = _ops_case(g, M, N, K, False, True, exact=False)
    C, Cpre = Window(M, N, torch.float32, "vec", C0), Window(M, N, torch.float32, "vec")
    n = _launches(L, lambda: ops_bf16.gemm(A, B, C.view, transB=True, alpha=0.5, beta=0.75, bias=bias, act=G.ACT_SILU,
                                           Cpre=Cpre.view))
    splits = G.sgemm_route(M, N, K)[3]
    assert n == 1 + (splits > 1), n
    f = dict(alpha=0.5, beta=0.75, C0=C0, bias=bias, act=G.ACT_SILU)
    ref = G.reference(_products(A, B, False, True), **f)
    for k, w in (("out", C), ("pre", Cpre)):
        ok, r, _ = G.check(w.view, *ref[k][:2], TAU)
        assert ok and w.outside_is_nan(), (k, r)
    WORST["ops_bf16_f32_fallback"] = {"out": G.check(C.view, *ref["out"][:2], TAU)[1]}
    # bf16 operands would be 2^-9 off: the rounded-operand oracle must not fit
    bad = G.reference(_products(A, B, False, True, rounded=True), **f)
    assert G.check(C.view, *bad["out"][:2], TAU)[1] >= 20 * TAU


@pytest.mark.parametrize("tB", [True, False])
def test_ops_bf16_shadow_operands_bit_identical_to_staged(L, ops_bf16, tB):
    M, N, K = 512, 384, 256
    assert G.ops_bf16_route(M, N, K) == "tc"
    g = torch.Generator().manual_seed(6 + tB)
    A, B, C0, bias = _ops_case(g, M, N, K, False, tB, exact=False)
    outs, counts = {}, {}
    for kind, ab, bb in (("staged", None, None), ("B", None, B.bfloat16()), ("AB", A.bfloat16(), B.bfloat16())):
        C = C0.clone()
        counts[kind] = _launches(L, lambda: ops_bf16.gemm(A, B, C, transB=tB, beta=0.75, bias=bias, act=G.ACT_RELU,
                                                          A_bf16=ab, B_bf16=bb))
        outs[kind] = C
    assert counts == {"staged": 3, "B": 2, "AB": 1}, counts      # casts of A and B, then one tensor-core launch
    assert torch.equal(_bits(outs["B"]), _bits(outs["staged"])) and torch.equal(_bits(outs["AB"]), _bits(outs["staged"]))
    ref = G.reference(_products(A, B, False, tB, rounded=True), beta=0.75, C0=C0, bias=bias, act=G.ACT_RELU)
    ok, r, _ = G.check(outs["staged"], *ref["out"][:2], TAU)
    WORST[f"ops_bf16_shadow_tB{int(tB)}"] = {"out": r}
    assert ok, r


def test_ops_bf16_shadow_with_unaligned_pitch_is_ignored(L, ops_bf16):
    M, N, K = 512, 384, 100                     # K % 8 != 0: the dense shadows' pitch cannot be read by TMA
    g = torch.Generator().manual_seed(7)
    A, B, C0, bias = _ops_case(g, M, N, K, False, True, exact=False)
    nan_a = torch.full((M, K), NAN, dtype=torch.bfloat16, device=DEV)
    nan_b = torch.full((N, K), NAN, dtype=torch.bfloat16, device=DEV)
    Cs, Cn = C0.clone(), C0.clone()
    n_staged = _launches(L, lambda: ops_bf16.gemm(A, B, Cs, transB=True, beta=0.75, bias=bias))
    n_shadow = _launches(L, lambda: ops_bf16.gemm(A, B, Cn, transB=True, beta=0.75, bias=bias, A_bf16=nan_a,
                                                  B_bf16=nan_b))
    assert n_staged == n_shadow == 3, (n_staged, n_shadow)
    assert torch.equal(_bits(Cn), _bits(Cs))
    ref = G.reference(_products(A, B, False, True, rounded=True), beta=0.75, C0=C0, bias=bias)
    assert G.check(Cn, *ref["out"][:2], TAU)[0]


@pytest.mark.parametrize("name", list(G.SGEMM_CASES))
@pytest.mark.parametrize("tA,tB", [(False, True), (False, False), (True, False), (True, True)])
def test_ops_fp32_sgemm_tiles_all_transposes(L, name, tA, tB):
    from tacorl_b200 import ops
    ops.set_precision("fp32")
    M, N, K, route = G.SGEMM_CASES[name]
    g = torch.Generator().manual_seed(M + N + K + 10 * tA + 20 * tB)
    A, B, C0, bias = _ops_case(g, M, N, K, tA, tB, exact=False)
    P = _products(A, B, tA, tB)
    worst = {}
    for en, f in (("silu_cpre_beta", dict(alpha=0.5, beta=0.75, C0=C0, bias=bias, act=G.ACT_SILU)),
                  ("relu_nan_c", dict(bias=bias, act=G.ACT_RELU))):
        C = Window(M, N, torch.float32, "vec", C0 if f.get("beta") else None)
        Cpre = Window(M, N, torch.float32, "vec")
        n = _launches(L, lambda: ops.gemm(A, B, C.view, transA=tA, transB=tB, alpha=f.get("alpha", 1.0),
                                          beta=f.get("beta", 0.0), bias=bias, act=f["act"], Cpre=Cpre.view))
        assert n == 1 + (route[3] > 1), (en, n, route)
        ref = G.reference(P, **f)
        for k, w in (("out", C), ("pre", Cpre)):
            ok, r, idx = G.check(w.view, *ref[k][:2], TAU)
            worst[f"{en}/{k}"] = r
            assert ok, (en, k, r, idx)
            assert w.outside_is_nan(), (en, k, "wrote outside [M, N]")
    WORST[f"{name}/tA{int(tA)}tB{int(tB)}"] = worst
