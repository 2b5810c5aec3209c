"""The bf16 LMP vision encoder (tacorl_lmp_encoder_{fwd,bwd} with PREC_BF16) checked stage by stage against the
teacher-forced fp64 oracle (tests/encoder_bf16_oracle.py), at the frame counts training runs.

Every stage, forward and backward, is checked per element on the kernel's own input of that stage: xs bit for bit;
y1, y2, dy3, dy2, dy1 within 1/2 bf16 ulp + TAU * S; y3, feat, smax, ssum, h4, emb, dh4, dfeat, the per-frame
temperature gradients and every parameter gradient within TAU * S.  The backward's intermediates are read from the
workspace after the call (`E.bwd_workspace`), which also shows that the zero margins of dy3 and dy1 are written.

Calibration: not yet measured on the B200.

The path each case claims is asserted: the fused FC head by the forward's launch count (the six conv-stack launches
plus one mlp_chain launch), each FC GEMM's operand precision by control 6 ("fc_precision_flipped" must fail on the
GEMM's own output: h4, emb, dW5, dW4, dfeat, and dh4 where it is kept), and xs rebuilt in the backward by one extra
launch, the rebuilt image's bits and bit-identical gradients against the same backward given the saved xs."""
import ctypes

import pytest
import torch

from tests import encoder_bf16_oracle as E
from tests.encoder_bf16_oracle import TAU
from tests.gpu_util import parity_report

pytestmark = pytest.mark.gpu

DEV = "cuda"
NAN = float("nan")
WORST = {}            # case -> {output: largest |err| / S}
CONTROLS = {}         # case -> {control: largest ratio over the outputs}
LAUNCHES = {}         # case -> (forward launches, fused FC head)
OUTS = ("y1", "y2", "y3", "feat", "smax", "ssum", "h4", "emb")


@pytest.fixture(scope="module")
def L():
    from tacorl_b200 import _lib
    _lib.lib()
    yield _lib
    parity_report("encoder_bf16_oracle", [{"tau": TAU, "worst_err_over_scale": WORST, "controls": CONTROLS,
                                           "forward_launches": LAUNCHES}])


def _vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def _same(a, b):
    return torch.equal(_bits(a), _bits(b))


def _launches(L, fn):
    torch.cuda.synchronize()
    n0 = L.launch_count()
    fn()
    torch.cuda.synchronize()
    return L.launch_count() - n0


class Case:
    """Inputs of one encoder call: weights at torch's default init scale, temperature `temp`, y3 channel 5 dead and
    channel 9 sharply peaked, uint8 or fp32 frames, pre-filled gradients when `acc`."""

    def __init__(self, N, H, W, u8, save_xs=True, acc=False, temp=0.7, seed=0):
        g = torch.Generator().manual_seed(seed or N * 7 + H * 3 + W)
        self.N, self.H, self.W, self.u8, self.save_xs, self.acc = N, H, W, u8, save_xs, int(acc)
        self.params = [p.to(DEV) for p in E.make_params(g, temp, dead=5, peaked=9)]
        self.x = E.make_input(g, N, H, W, u8).to(DEV)
        self.d_emb = torch.randn(N, E.LATENT, generator=g).to(DEV)
        self.pre = [torch.randn(p.shape, generator=g).to(DEV) for p in self.params] if acc else None
        self.H1, self.W1 = (H - 8) // 4 + 1, (W - 8) // 4 + 1
        self.H2, self.W2 = (self.H1 - 4) // 2 + 1, (self.W1 - 4) // 2 + 1
        self.H3, self.W3 = self.H2 - 2, self.W2 - 2
        self.norm = (1, E.NORM_SCALE, E.NORM_SHIFT) if u8 else (0, 1.0, 0.0)
        self.fc = E.fc_paths(N, E.HIDDEN, E.LATENT, acc)

    def ws(self, L, backward, fill):
        n = L.query("tacorl_lmp_encoder_ws_bytes", self.N, self.H, self.W, E.HIDDEN, E.LATENT, backward)
        return torch.full((int(n),), fill, dtype=torch.uint8, device=DEV)

    def fwd(self, L, save=True, fill=0xFF):
        N, bf = self.N, torch.bfloat16
        o = {"emb": torch.full((N, E.LATENT), NAN, device=DEV)}
        if save:
            o.update(y1=torch.full((N, self.H1, self.W1, 32), NAN, device=DEV, dtype=bf),
                     y2=torch.full((N, self.H2, self.W2, 64), NAN, device=DEV, dtype=bf),
                     y3=torch.full((N, self.H3, self.W3, 64), NAN, device=DEV),
                     feat=torch.full((N, 128), NAN, device=DEV), smax=torch.full((N, 64), NAN, device=DEV),
                     ssum=torch.full((N, 64), NAN, device=DEV), h4=torch.full((N, E.HIDDEN), NAN, device=DEV))
            if self.save_xs:
                o["xs"] = torch.full((N, self.H1 + 1, self.W1 + 1, 64), NAN, device=DEV, dtype=bf)
        ws = self.ws(L, 0, fill)
        o["launches"] = _launches(L, lambda: L.call(
            "tacorl_lmp_encoder_fwd", _vp(self.x), *self.norm, N, self.H, self.W, L.ptr_array(self.params), E.HIDDEN,
            E.LATENT, _vp(o.get("y1")), _vp(o.get("y2")), _vp(o.get("y3")), _vp(o.get("feat")), _vp(o.get("smax")),
            _vp(o.get("ssum")), _vp(o.get("h4")), _vp(o["emb"]), _vp(o.get("xs")), _vp(ws), ws.numel(), L.PREC_BF16,
            L.stream()))
        return o

    def bwd(self, L, f, xs=None, fill=0xFF):
        grads = ([p.clone() for p in self.pre] if self.acc else [torch.full_like(p, NAN) for p in self.params])
        ws = self.ws(L, 1, fill)
        k = _launches(L, lambda: L.call(
            "tacorl_lmp_encoder_bwd", _vp(self.x), *self.norm, self.N, self.H, self.W, L.ptr_array(self.params),
            E.HIDDEN, E.LATENT, _vp(f["y1"]), _vp(f["y2"]), _vp(f["y3"]), _vp(f["feat"]), _vp(f["smax"]),
            _vp(f["ssum"]), _vp(f["h4"]), _vp(self.d_emb), L.ptr_array(grads), self.acc, _vp(xs), _vp(ws), ws.numel(),
            L.PREC_BF16, L.stream()))
        inter = E.bwd_workspace(ws, self.N, self.H, self.W, E.HIDDEN, xs is not None)
        return dict(zip(E.PARAMS, grads)), k, inter

    def xs_want(self):
        return E.s2d(self.x, E.NORM_SCALE, E.NORM_SHIFT) if self.u8 else E.s2d(self.x)

    def oracle(self, f, inter, control=None):
        xs = f.get("xs") if self.save_xs else self.xs_want()
        a = (self.params, xs, f["y1"], f["y2"], f["y3"], f["feat"], f["h4"])
        ref = E.fwd(*a, self.fc, control)
        ref.update(E.bwd(*a, self.d_emb, self.fc, inter, self.pre, control))
        return ref


def _assert_ok(tag, got, ref):
    res = E.check_all(got, ref, TAU)
    WORST[tag] = {k: r[1] for k, r in res.items()}
    bad = {k: f"{r[1]:.3e}" for k, r in res.items() if not r[0]}
    assert not bad, f"{tag}: max |err|/S over TAU = {TAU:g}: {bad}"
    return res


def _got(f, grads, inter):
    got = {k: f[k] for k in OUTS}
    got.update(grads)
    got.update({k: inter[k] for k in ("dh4", "dfeat", "dtau", "dy3", "dy2", "dy1")})
    return got


def _run(L, case, tag):
    f = case.fwd(L)
    grads, _, inter = case.bwd(L, f, f.get("xs"))
    torch.cuda.synchronize()
    xs = f["xs"] if case.save_xs else inter["xs"]
    assert _same(xs, case.xs_want()), f"{tag}: space-to-depth image differs from the oracle's"
    assert all(int(_bits(m).abs().max()) == 0 for m in inter["margins"]), f"{tag}: dy3 / dy1 margin not zeroed"
    got = _got(f, grads, inter)
    ref = case.oracle(f, inter)
    _assert_ok(tag, got, ref)
    LAUNCHES[tag] = (f["launches"], case.fc["fc1"] == "fused")
    # control 6 on this case's own data: every FC GEMM's operand precision is the claimed one
    r = E.check_all(got, case.oracle(f, inter, "fc_precision_flipped"), TAU)
    outs = ["h4", "emb", "W5", "W4", "dfeat"] + ([] if case.fc["dh4"] == "fused" else ["dh4"])
    CONTROLS.setdefault(tag, {})["fc_precision_flipped"] = {k: r[k][1] for k in outs}
    assert all(r[k][1] >= 20 * TAU for k in outs), (tag, {k: r[k][1] for k in outs})
    return f, grads, got, ref


# (N, H, W, uint8, xs saved): what each exercises
CASES = [
    (1, 84, 84, False, True),       # one frame, fp32 input
    (3, 128, 128, True, True),
    (2, 150, 200, False, False),    # H not a multiple of 4, non-square, xs rebuilt in the backward
    (256, 84, 84, True, True),      # last fused-FC size
    (257, 84, 84, True, True),      # non-fused FC head, every FC GEMM fp32
    (777, 84, 84, True, True),      # mixed FC paths, ragged K on the transA operands
    (2048, 84, 84, True, True),     # every FC GEMM on the tensor cores
    (1024, 84, 84, True, True),     # bench.py's gripper view
    (1024, 200, 200, True, True),   # bench.py's PlayLMP static view
]


@pytest.mark.parametrize("N,H,W,u8,save_xs", CASES, ids=lambda v: str(v))
def test_encoder_matches_oracle(L, N, H, W, u8, save_xs):
    case = Case(N, H, W, u8, save_xs)
    tag = f"N{N} {H}x{W} {'u8' if u8 else 'f32'}{'' if save_xs else ' xs-rebuilt'}"
    f, grads, _, _ = _run(L, case, tag)
    if not save_xs:      # the backward rebuilt xs: one more launch than given the oracle's (bit-identical) xs
        xs = case.xs_want()
        g2, k2, _ = case.bwd(L, f, xs)
        g1, k1, _ = case.bwd(L, f, None)
        torch.cuda.synchronize()
        assert k1 == k2 + 1, (k1, k2)
        assert all(_same(g1[k], g2[k]) and _same(g1[k], grads[k]) for k in E.PARAMS)


@pytest.mark.parametrize("N", [3, 300])
def test_encoder_accumulate_matches_oracle(L, N):
    """accumulate = 1: the non-fused FC head at any size and beta = 1 in every weight-gradient reduction."""
    case = Case(N, 84, 84, True, acc=True, temp=1.3)
    assert case.fc["dW4"] != "fused"
    _run(L, case, f"N{N} 84x84 u8 accumulate")


def test_encoder_small_temperature_matches_oracle(L):
    """temperature 0.25: exponent arguments down to about -100 in the peaked channel."""
    _run(L, Case(4, 84, 84, True, temp=0.25), "N4 84x84 u8 temperature 0.25")


CONV_STACK_LAUNCHES = 6      # weight packing, space-to-depth, conv1, conv2, conv3, soft-argmax


def test_fused_fc_head_is_one_launch(L):
    """Up to 256 frames the forward is the conv stack plus exactly one launch (the fused FC head); at 257 frames the
    head is two separate fp32 GEMMs, which take more than one launch."""
    k1 = Case(1, 84, 84, True).fwd(L)["launches"]
    k256 = Case(256, 84, 84, True).fwd(L)["launches"]
    k257 = Case(257, 84, 84, True).fwd(L)["launches"]
    assert k1 == k256 == CONV_STACK_LAUNCHES + 1 and k257 > k256, (k1, k256, k257)


def test_workspace_contents_do_not_matter(L):
    """Once with the workspace filled with 0xFF bytes, once with zeros: every output, saved tensor and gradient bit
    for bit the same (the encoder has no float atomics: a difference is a read of uninitialised memory)."""
    case = Case(777, 84, 84, True)
    fa = case.fwd(L, fill=0xFF)
    ga, _, _ = case.bwd(L, fa, fa["xs"], fill=0xFF)
    fb = case.fwd(L, fill=0)
    gb, _, _ = case.bwd(L, fb, fb["xs"], fill=0)
    torch.cuda.synchronize()
    for k in OUTS + ("xs",):
        assert _same(fa[k], fb[k]), k
    for k in E.PARAMS:
        assert _same(ga[k], gb[k]), k


@pytest.mark.parametrize("N,H,W", [(3, 128, 128), (1024, 84, 84)])
def test_inference_forward_matches_training_forward(L, N, H, W):
    """save = False (y1 .. h4 and xs NULL, all in the workspace): the same emb bits as the training forward."""
    case = Case(N, H, W, True)
    a = case.fwd(L, save=True)
    b = case.fwd(L, save=False)
    torch.cuda.synchronize()
    assert _same(a["emb"], b["emb"])


def test_model_level_op_is_the_verified_abi_chain(L):
    """ops.lmp_encoder under set_precision("bf16") makes exactly the ABI calls checked above: emb and every gradient
    bit for bit."""
    from tacorl_b200 import ops
    case = Case(64, 84, 84, True)
    f = case.fwd(L)
    grads, _, _ = case.bwd(L, f, f["xs"])
    ops.set_precision("bf16")
    try:
        ps = [p.clone().requires_grad_(True) for p in case.params]
        emb = ops.lmp_encoder(case.x, ps, norm=(0.5, 0.5))
        emb.backward(case.d_emb)
    finally:
        ops.set_precision("fp32")
    torch.cuda.synchronize()
    assert _same(emb.detach(), f["emb"])
    for k, p in zip(E.PARAMS, ps):
        assert _same(p.grad, grads[k]), k


def test_oracle_check_catches_subtle_errors_on_kernel_data(L):
    """On kernel data: the unaltered oracle passes, every control fails by at least 20 * TAU, and so does a one-ulp
    change of one element of each bf16 output (xs: any change breaks bit equality)."""
    case = Case(3, 84, 84, True, acc=True, temp=1.3)
    f = case.fwd(L)
    grads, _, inter = case.bwd(L, f, f["xs"])
    torch.cuda.synchronize()
    got = _got(f, grads, inter)
    ref = case.oracle(f, inter)
    _assert_ok("controls case N3 84x84 u8 accumulate", got, ref)
    ratios = {}
    for control in E.CONTROLS:
        r = E.check_all(got, case.oracle(f, inter, control), TAU)
        ratios[control] = max(v[1] for v in r.values())
    CONTROLS["controls case N3 84x84 u8 accumulate"] = ratios
    assert all(v >= 20 * TAU for v in ratios.values()), ratios
    for name in E.BF16_OUT:
        want, scale = ref[name][:2]
        ok, ratio, _ = E.check(E.bump_one_ulp(got[name], want, scale), want, scale, TAU, bf16=True)
        assert not ok and ratio >= 20 * TAU, (name, ratio)
    xs = f["xs"].clone()
    xs.view(-1)[7] = xs.view(-1)[7] + 1.0
    assert not _same(xs, case.xs_want())
