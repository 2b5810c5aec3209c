"""The teacher-forced bf16 encoder oracle (tests/encoder_bf16_oracle.py) checked on the CPU before any GPU is involved:
  - its fp64 formulas (no bf16 rounding, bf16-exact inputs) reproduce oracle.tacorl_oracle.lmp_encoder and the
    autograd gradients of every parameter;
  - a torch emulation of the kernels' arithmetic (bf16 operands, fp32 accumulation, bf16 roundings where the kernels
    round) passes the check at the tolerance the GPU tests use;
  - every discrimination control fails it by at least 20x that tolerance, and so does a one-ulp change of one element
    of each bf16 output."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch.nn.grad import conv2d_input, conv2d_weight

from oracle import tacorl_oracle as O
from tests import encoder_bf16_oracle as E
from tests.encoder_bf16_oracle import TAU

NAMES = ["model.0.weight", "model.0.bias", "model.2.weight", "model.2.bias", "model.4.weight", "model.4.bias",
         "model.6.temperature", "fc_layers.0.weight", "fc_layers.0.bias", "fc_layers.3.weight", "fc_layers.3.bias"]
HIDDEN, LATENT = E.HIDDEN, E.LATENT
NORM_SCALE, NORM_SHIFT = E.NORM_SCALE, E.NORM_SHIFT
make_params, make_input = E.make_params, E.make_input


def _bf(t):
    return t.bfloat16().float()


def emulate(params, x, fc, d_emb, pre=None, exact=False):
    """The kernels' arithmetic in torch: fp32 accumulation over bf16 operands, bf16 roundings of y1, y2, dy3, dy2, dy1
    and of tensor-core FC operands.  exact: float64 everywhere and no rounding beyond the bf16 space-to-depth image.
    Returns the kernel tensors (NHWC activations; "ws": the backward's intermediates) and the gradients in PARAMS
    order."""
    dt = torch.float64 if exact else torch.float32
    rnd = (lambda t: t) if exact else _bf
    W1, b1, W2, b2, W3, b3, temp, W4, b4, W5, b5 = [p.to(dt) for p in params]
    xs = E.s2d(x, NORM_SCALE, NORM_SHIFT) if x.dtype == torch.uint8 else E.s2d(x)
    img = E.unpack_xs(xs).to(dt)
    w1, w2, w3 = rnd(W1), rnd(W2), rnd(W3)
    y1 = rnd(torch.relu(F.conv2d(img, w1, b1, stride=4)))
    y2 = rnd(torch.relu(F.conv2d(y1, w2, b2, stride=2)))
    y3 = torch.relu(F.conv2d(y2, w3, b3))
    N, C, H3, W3s = y3.shape
    inv_t = 1 / temp
    z = y3.permute(0, 2, 3, 1).reshape(N, H3 * W3s, C) * inv_t
    m = z.amax(1, keepdim=True)
    e = torch.exp(z - m)
    s = e.sum(1, keepdim=True)
    pos = torch.arange(H3 * W3s, dtype=dt)
    col, row = (pos % W3s).view(1, -1, 1), torch.div(pos, W3s, rounding_mode="floor").view(1, -1, 1)
    fx, fy = (e * col).sum(1) / s[:, 0], (e * row).sum(1) / s[:, 0]
    feat = torch.stack([fx, fy], -1).reshape(N, 2 * C)
    op = {k: (_bf if (v == "tc" and not exact) else (lambda t: t)) for k, v in fc.items()}
    h4 = torch.relu(op["fc1"](feat) @ op["fc1"](W4).t() + b4)
    emb = op["fc2"](h4) @ op["fc2"](W5).t() + b5
    g = d_emb.to(dt)
    gr = [None] * 11
    gr[9] = op["dW5"](g).t() @ op["dW5"](h4)
    gr[10] = g.sum(0)
    dh4 = (op["dh4"](g) @ op["dh4"](W5)) * (h4 > 0)
    gr[8] = dh4.sum(0)
    gr[7] = op["dW4"](dh4).t() @ op["dW4"](feat)
    dfeat = op["dfeat"](dh4) @ op["dfeat"](W4)
    p = e / s
    gx, gy = dfeat.reshape(N, C, 2)[..., 0].unsqueeze(1), dfeat.reshape(N, C, 2)[..., 1].unsqueeze(1)
    dotg = gx * fx.unsqueeze(1) + gy * fy.unsqueeze(1)
    dz = p * (gx * col + gy * row - dotg)
    yv = y3.permute(0, 2, 3, 1).reshape(N, H3 * W3s, C)
    dtau = -(dz * yv).sum((1, 2)) * inv_t * inv_t
    gr[6] = dtau.sum().reshape(1)
    dy3 = rnd((dz * inv_t * (yv > 0)).reshape(N, H3, W3s, C).permute(0, 3, 1, 2))
    gr[4], gr[5] = conv2d_weight(y2, W3.shape, dy3), dy3.sum((0, 2, 3))
    dy2 = rnd(conv2d_input(y2.shape, w3, dy3) * (y2 > 0))
    gr[2], gr[3] = conv2d_weight(y1, W2.shape, dy2, stride=2), dy2.sum((0, 2, 3))
    dy1 = rnd(conv2d_input(y1.shape, w2, dy2, stride=2) * (y1 > 0))
    gr[0], gr[1] = conv2d_weight(img, W1.shape, dy1, stride=4), dy1.sum((0, 2, 3))
    if pre is not None:
        gr = [a + b.to(dt) for a, b in zip(gr, pre)]
    nhwc = lambda t: t.permute(0, 2, 3, 1).contiguous()     # noqa: E731
    k = {"xs": xs, "y1": nhwc(y1), "y2": nhwc(y2), "y3": nhwc(y3), "feat": feat, "smax": m.reshape(N, C),
         "ssum": s.reshape(N, C), "h4": h4, "emb": emb}
    k["ws"] = {"dh4": dh4, "dfeat": dfeat, "dtau": dtau, "dy3": nhwc(dy3), "dy2": nhwc(dy2), "dy1": nhwc(dy1)}
    if not exact:
        k["y1"], k["y2"] = k["y1"].bfloat16(), k["y2"].bfloat16()
        for n in ("dy3", "dy2", "dy1"):
            k["ws"][n] = k["ws"][n].bfloat16()
    return k, gr


def oracle(params, k, d_emb, fc, pre=None, control=None):
    ref = E.fwd(params, k["xs"], k["y1"], k["y2"], k["y3"], k["feat"], k["h4"], fc, control)
    ref.update(E.bwd(params, k["xs"], k["y1"], k["y2"], k["y3"], k["feat"], k["h4"], d_emb, fc, k["ws"], pre, control))
    return ref


def got_of(k, gr):
    got = {n: k[n] for n in ("y1", "y2", "y3", "feat", "smax", "ssum", "h4", "emb")}
    got.update(dict(zip(E.PARAMS, gr)))
    got.update(k["ws"])
    return got


def test_exact_formulas_reproduce_the_fp64_reference():
    g = torch.Generator().manual_seed(3)
    params = [_bf(p) for p in make_params(g)]
    x = _bf(make_input(g, 2, 84, 84, False))
    d_emb = torch.randn(2, LATENT, generator=g)
    fc = E.fc_paths(2, HIDDEN, LATENT)
    k, _ = emulate(params, x, fc, d_emb, exact=True)
    P = {n: p.double().requires_grad_(True) for n, p in zip(NAMES, params)}
    emb = O.lmp_encoder(P, "", x.double())
    (emb * d_emb.double()).sum().backward()
    ref = oracle(params, k, d_emb, fc)
    assert torch.allclose(ref["emb"][0], emb.detach(), rtol=1e-12, atol=1e-12)
    feat = O.spatial_softargmax(O.lmp_encoder_convs(P, "", x.double()), P["model.6.temperature"])
    assert torch.allclose(ref["feat"][0], feat.detach(), rtol=1e-12, atol=1e-12)
    for name, pn in zip(E.PARAMS, NAMES):
        want = P[pn].grad
        got = ref[name][0].reshape(want.shape)
        err = float((got - want).abs().max() / (want.abs().max() + 1e-300))
        assert err < 1e-11, (name, err)


CASES = [  # (N, H, W, u8, temperature, fc override, accumulate)
    (2, 84, 84, True, 0.7, None, False),
    (2, 150, 200, False, 0.7, None, False),
    (2, 84, 84, True, 1.3, "tc", True),
    (2, 84, 84, False, 0.25, "f32", False),
]


@pytest.mark.parametrize("N,H,W,u8,temp,fcall,acc", CASES)
def test_emulated_kernel_passes_and_controls_fail(N, H, W, u8, temp, fcall, acc):
    g = torch.Generator().manual_seed(N * 1000 + H + W)
    params = make_params(g, temp, dead=5, peaked=9)
    x = make_input(g, N, H, W, u8)
    d_emb = torch.randn(N, LATENT, generator=g)
    fc = E.fc_paths(N, HIDDEN, LATENT, acc)
    if fcall is not None:
        fc = {kk: fcall for kk in fc}
    pre = [torch.randn(p.shape, generator=g) for p in params] if acc else None
    k, gr = emulate(params, x, fc, d_emb, pre)
    got = got_of(k, gr)
    ref = oracle(params, k, d_emb, fc, pre)
    res = E.check_all(got, ref, TAU)
    assert all(r[0] for r in res.values()), {kk: r[1] for kk, r in res.items()}
    # the emulation sits well inside TAU: the bar has head room for the kernels' own summation orders
    assert max(r[1] for r in res.values()) < TAU / 4, {kk: r[1] for kk, r in res.items()}
    assert torch.equal(k["xs"].view(torch.int16), (E.s2d(x, NORM_SCALE, NORM_SHIFT) if u8 else E.s2d(x)).view(torch.int16))
    # the dead channel: uniform softmax, zero gradient through it
    assert float(k["y3"][..., 5].abs().max()) == 0
    for control in E.CONTROLS:
        if control == "accumulate_ignored" and not acc:
            continue
        r = E.check_all(got, oracle(params, k, d_emb, fc, pre, control), TAU)
        worst = max(v[1] for v in r.values())
        assert worst >= 20 * TAU, (control, {kk: v[1] for kk, v in r.items()})
        if control == "fc_precision_flipped":     # each FC GEMM's precision is observable on its own output
            outs = ["h4", "emb", "dfeat", "W5"] + ([] if fc["dh4"] == "fused" else ["dh4"])
            assert all(r[o][1] >= 20 * TAU for o in outs), {o: r[o][1] for o in outs}
    for name in E.BF16_OUT:
        want, scale = ref[name][:2]
        ok, ratio, _ = E.check(E.bump_one_ulp(got[name], want, scale), want, scale, TAU, bf16=True)
        assert not ok and ratio >= 20 * TAU, (name, ratio)


def test_s2d_layout_and_u8_rounding():
    g = torch.Generator().manual_seed(0)
    x = make_input(g, 1, 84, 88, True)
    xs = E.s2d(x, NORM_SCALE, NORM_SHIFT)
    assert xs.shape == (1, 21, 22, 64)
    n, Y, X, py, px, c = 0, 3, 5, 2, 1, 2
    v = np.float32(np.float32(x[n, c, 4 * Y + py, 4 * X + px].item()) * np.float32(NORM_SCALE) + np.float32(NORM_SHIFT))
    assert xs[n, Y, X, py * 12 + px * 3 + c].item() == torch.tensor(float(v)).bfloat16().item()
    assert float(xs[..., 48:].abs().max()) == 0
    assert torch.equal(E.unpack_xs(xs)[0, c, 4 * Y + py, 4 * X + px].reshape(1), xs[n, Y, X, py * 12 + px * 3 + c].double().reshape(1))


def test_fc_paths_follow_the_per_gemm_rule():
    assert set(E.fc_paths(256, 256, 32).values()) == {"fused"}
    assert set(E.fc_paths(257, 256, 32).values()) == {"f32"}
    assert E.fc_paths(3, 256, 32, accumulate=True) == {"fc1": "fused", "fc2": "fused", "dW5": "f32", "dh4": "f32",
                                                        "dW4": "f32", "dfeat": "f32"}
    assert E.fc_paths(1024, 256, 32) == {"fc1": "tc", "fc2": "f32", "dW5": "f32", "dh4": "f32", "dW4": "tc", "dfeat": "tc"}
    assert set(E.fc_paths(2048, 256, 32).values()) == {"tc"}


def test_check_allowances():
    want = torch.tensor([1.0, 2.0, 0.0], dtype=torch.float64)
    s = torch.ones(3, dtype=torch.float64)
    got = torch.tensor([1.0 + 2.0 ** -8, 2.0, 0.0])          # half a bf16 ulp of 1.0 off
    assert not E.check(got, want, s, 1e-5)[0]
    assert E.check(got, want, s, 1e-5, bf16=True)[0]
    b = E.bump_one_ulp(torch.tensor([1.0, 2.0, 0.5]).bfloat16(), want, s)
    assert float(b[1]) == 2.0 + 2.0 ** -6                      # |2| against its scale is the largest: ulp(2..4) = 2^-6
    u = E.bwd_workspace(torch.zeros(1 << 28, dtype=torch.uint8), 2, 84, 84, 256, False)
    assert u["dy3"].shape == (2, 7, 7, 64) and u["dy1"].shape == (2, 20, 20, 32) and u["xs"].shape == (2, 21, 21, 64)
    assert u["dfeat"].data_ptr() - u["dh4"].data_ptr() == 2 * 256 * 4 and [m.numel() for m in u["margins"]] == [2 * 2 * 9 * 64, 2 * 7 * 2 * 64, 2 * 21 * 32, 2 * 20 * 32]
