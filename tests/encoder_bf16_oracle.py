"""Teacher-forced fp64 oracle of the bf16 LMP vision encoder (tacorl_lmp_encoder_{fwd,bwd} with PREC_BF16:
enc_fwd_tc / enc_bwd_tc in encoder.cu).

Forward.  Every stage's input is a tensor the caller owns and reads back after the call (marked K): the bf16
space-to-depth image `xs`, bf16 `y1` and `y2`, fp32 `y3`, `feat` and `h4`.  So each stage is checked on the kernel's
own input, and the only error left in it is the kernel's fp32 arithmetic:
  xs    = s2d(rne(x)), or s2d(rne(fp32(u8 * scale + shift))) for uint8 frames: bit equality;
  y1    = relu(conv1(xs_K, rne(W1)) + b1)        (bf16 output: |got - want| <= 1/2 ulp_bf16(want) + TAU * S)
  y2    = relu(conv2(y1_K, rne(W2)) + b2)        (bf16 output)
  y3    = relu(conv3(y2_K, rne(W3)) + b3)        (fp32)
  feat, smax, ssum = spatial soft-argmax of y3_K / temperature; x is the column, y the row.  smax is the largest
          y3 / temperature of the (frame, channel), ssum = sum exp(y3 / temperature - smax)
  h4    = relu(feat_K W4^T + b4), emb = h4_K W5^T + b5, fp32 operands on the fused FC head and on GEMMs below 2^24
          multiply-adds, rne operands on the tensor-core GEMMs (`fc_paths`).

Backward, teacher-forced the same way.  Its intermediates are not outputs of the ABI, but they stay in the
caller's workspace after the call, at offsets fixed by enc_bwd_tc's carve order (`bwd_workspace` reads them): the
fp32 dh4 (non-fused FC head only), dfeat and the per-frame temperature gradients, and the bf16 dy3, dy2 and dy1 at the
pitches the kernels use.  So every backward stage is checked on the kernel's own input of that stage too:
  dh4   = (op(d_emb) op(W5)) * [h4_K > 0]              (fp32; op = rne on tensor-core GEMMs, identity on fp32 ones)
  dfeat = op(dh4_K) op(W4),  dW4 = op(dh4_K)^T op(feat_K),  db4 = sum dh4_K,  dW5 = op(d_emb)^T op(h4_K), db5 = sum d_emb
          (the fused fp32 head keeps dh4 in registers: there dfeat / dW4 / db4 take the oracle's fp64 dh4 and its scale)
  dy3   = [y3_K > 0] * p (gx (col - fx_K) + gy (row - fy_K)) / temperature, (gx, gy) from dfeat_K     (bf16 output)
  dtau  = -sum dz * y3_K / temperature^2 per frame; d temperature = sum over frames
  dW3, db3 from dy3_K and y2_K;  dy2 = [y2_K > 0] * conv3_data_grad(dy3_K, rne(W3))                 (bf16 output)
  dW2, db2 from dy2_K and y1_K;  dy1 = [y1_K > 0] * conv2_data_grad(dy2_K, rne(W2))                 (bf16 output)
  dW1, db1 from dy1_K and xs_K.
Conv bias gradients are the column sums of the bf16 gradient the weight-gradient kernels consume (their extra MMA
against an all-ones operand).  With accumulate = 1 the pre-filled value is added.  No stage consumes a value the oracle
rounded itself, so a rounding boundary cannot fall between kernel and oracle anywhere but in a checked bf16 output,
where the half-ulp allowance covers it: the backward is held to the same bar as the forward.

Scale S of an output is the first-order bound of its fp32 evaluation error: the same contraction on absolute values,
with an fp32 intermediate's scale carried into its consumers (only on the fused FC head).  In the soft-argmax, the
exponent's argument error is proportional to |y / temperature| (the products y * (1 / temperature) are rounded), so
each probability weighs 1 + |z| + |max z| there (not for the maximum itself, whose exponent is exactly 0).

`control` alters the oracle the way a subtle kernel bug would (the tests assert that the check then fails):
  "conv_w_fp32"            conv weights not rounded to bf16;
  "conv1_taps_transposed"  conv1's taps transposed (ky <-> kx);
  "dy2_no_relu_mask"       conv3's data gradient without y2's ReLU mask;
  "conv2_parity_swap"      conv2's data gradient with the (0, 1) and (1, 0) stride-parity classes' taps swapped;
  "softargmax_xy_swapped"  the soft-argmax's x (column) and y (row) coordinates swapped;
  "fc_precision_flipped"   every FC GEMM with the opposite operand precision (fp32 <-> rne);
  "accumulate_ignored"     the pre-filled gradients are not added (accumulate = 1);
  "dy_unrounded"           the weight and bias gradients consume unrounded dy3 / dy2 / dy1 instead of the bf16 ones;
  "dy_truncated"           dy3 / dy2 / dy1 rounded toward zero instead of to nearest even;
  "bias_from_fp32_dy"      the conv bias gradients summed from the unrounded dy instead of the bf16 one;
  "dy1_scaled"             dy1 scaled by 1 + 2^-9 before rounding.
"""
import torch
import torch.nn.functional as F
from torch.nn.grad import conv2d_input, conv2d_weight

CONTROLS = ("conv_w_fp32", "conv1_taps_transposed", "dy2_no_relu_mask", "conv2_parity_swap", "softargmax_xy_swapped",
            "fc_precision_flipped", "accumulate_ignored", "dy_unrounded", "dy_truncated", "bias_from_fp32_dy",
            "dy1_scaled")
# per-element bar |got - want| <= TAU * S (+ 1/2 ulp_bf16(want) on bf16 outputs);
# calibration: tests/test_gpu_encoder_bf16_oracle.py
TAU = 1e-5
PARAMS = ("W1", "b1", "W2", "b2", "W3", "b3", "temp", "W4", "b4", "W5", "b5")     # state_dict order
FC_GEMMS = ("fc1", "fc2", "dW5", "dh4", "dW4", "dfeat")
TC_MACS = 1 << 24        # gemm_tc_from_f32: tensor cores from M * N * K >= 2^24 multiply-adds
FUSED_MAX = 256          # fc_fused_ok: frames up to which the FC head is one fused fp32 kernel each way


def rne(t):
    """The bf16 value the kernels feed the tensor cores (round to nearest even), as float64."""
    return t.float().bfloat16().double()


def ulp_bf16(t):
    """bf16 ulp of |t| (float64): 2^(exponent - 7); the smallest normal's ulp for zeros."""
    e = torch.frexp(t.double().abs().clamp_min(2.0 ** -126))[1]
    return torch.ldexp(torch.ones_like(t, dtype=torch.float64), e - 8)


def fc_paths(N, hidden, latent, accumulate=False):
    """Path of each FC GEMM: "fused" (one fp32 mlp_chain kernel), "f32" (SIMT) or "tc" (rne operands).  The backward
    never fuses with accumulate = 1."""
    fused_f = N <= FUSED_MAX and hidden % 4 == 0 and hidden <= 256 and latent <= 256
    fused_b = fused_f and not accumulate
    macs = {"fc1": N * hidden * 128, "fc2": N * latent * hidden, "dW5": latent * hidden * N, "dh4": N * hidden * latent,
            "dW4": hidden * 128 * N, "dfeat": N * 128 * hidden}
    out = {}
    for k, m in macs.items():
        fused = fused_f if k in ("fc1", "fc2") else fused_b
        out[k] = "fused" if fused else ("tc" if m >= TC_MACS else "f32")
    return out


# ------------------------------------------------------------------------------------------ case inputs
HIDDEN, LATENT = 256, 32       # LMPVisionEncoder's FC head
# (u8 / 255 - 0.5) / 0.5 as LMPEncoderFn passes it to the kernels: u8 * scale + shift with fp32 scale and shift
NORM_SCALE = float(torch.tensor(1.0 / (255.0 * 0.5), dtype=torch.float32))
NORM_SHIFT = float(torch.tensor(-0.5 / 0.5, dtype=torch.float32))


def make_params(g, temp=0.7, dead=None, peaked=None):
    """Weights at torch's default init scale (U(+-1/sqrt(fan_in)) for Conv2d and Linear weights and biases).
    dead: a y3 channel pushed far below zero (uniform softmax, zero gradient); peaked: one with a large bias and
    four times the weights (large exponent arguments)."""
    shapes = [((32, 3, 8, 8), 192), ((32,), 192), ((64, 32, 4, 4), 512), ((64,), 512), ((64, 64, 3, 3), 576), ((64,), 576),
              None, ((HIDDEN, 128), 128), ((HIDDEN,), 128), ((LATENT, HIDDEN), HIDDEN), ((LATENT,), HIDDEN)]
    out = []
    for s in shapes:
        if s is None:
            out.append(torch.tensor([temp]))
            continue
        shape, fan = s
        out.append((torch.rand(*shape, generator=g) * 2 - 1) / fan ** 0.5)
    if dead is not None:
        out[5][dead] = -50.0
    if peaked is not None:
        out[4][peaked] *= 4
        out[5][peaked] = 8.0
    return out


def make_input(g, N, H, W, u8):
    if u8:
        return torch.randint(0, 256, (N, 3, H, W), generator=g, dtype=torch.uint8)
    return torch.rand(N, 3, H, W, generator=g) * 2 - 1


def _d(t):
    return t.detach().double()


def _nchw(t):
    return _d(t).permute(0, 3, 1, 2)


# ------------------------------------------------------------------------------------------ space-to-depth
def s2d(x, scale=None, shift=None):
    """The bf16 space-to-depth image the kernels build: (N, H1+1, W1+1, 64), channel (py*4 + px)*3 + c of pixel (Y, X)
    = x[n, c, 4Y+py, 4X+px], channels 48..63 zero.  uint8 frames: u8 * scale + shift is exact in fp64, so rounding it
    to fp32 and then to bf16 is what fmaf followed by __floats2bfloat16_rn does.  Returns bf16 (bit-comparable)."""
    N, C, H, W = x.shape
    SH, SW = (H - 8) // 4 + 2, (W - 8) // 4 + 2
    if x.dtype == torch.uint8:
        v = (x.double() * scale + shift).float()
    else:
        v = x.float()
    v = v[:, :, :4 * SH, :4 * SW].reshape(N, 3, SH, 4, SW, 4).permute(0, 2, 4, 3, 5, 1).reshape(N, SH, SW, 48)
    out = torch.zeros(N, SH, SW, 64, dtype=torch.bfloat16, device=x.device)
    out[..., :48] = v.bfloat16()
    return out


def unpack_xs(xs):
    """(N, SH, SW, 64) space-to-depth image -> the (N, 3, 4 SH, 4 SW) float64 image it holds."""
    N, SH, SW, _ = xs.shape
    v = _d(xs[..., :48]).reshape(N, SH, SW, 4, 4, 3)
    return v.permute(0, 5, 1, 3, 2, 4).reshape(N, 3, 4 * SH, 4 * SW)


# ------------------------------------------------------------------------------------------ helpers
def _conv(x, w, stride, b=None):
    """(value, scale) of relu-less conv2d(x, w) + b."""
    v = F.conv2d(x, w, stride=stride)
    s = F.conv2d(x.abs(), w.abs(), stride=stride)
    if b is not None:
        v, s = v + b.view(1, -1, 1, 1), s + b.abs().view(1, -1, 1, 1)
    return v, s


def _conv_w(control, w):
    return _d(w) if control == "conv_w_fp32" else rne(w)


def _w1(control, w):
    w = _conv_w(control, w)
    return w.transpose(2, 3) if control == "conv1_taps_transposed" else w


def _fc_op(path, control, exact=False):
    """Operand map of one FC GEMM: identity on fp32 paths, rne on tensor cores (opposite under the control)."""
    tc = path == "tc"
    if control == "fc_precision_flipped":
        tc = not tc
    return rne if (tc and not exact) else (lambda t: t)


def _softmax(y3, temp):
    """fp64 soft-argmax pieces of y3 (N, H3, W3, C): p (N, P, C), z = y3 / temp, m = max z, a = the weights of the
    exponent's argument error, coordinates (col, row) per position."""
    N, H3, W3, C = y3.shape
    z = _d(y3).reshape(N, H3 * W3, C) / temp
    m = z.amax(1, keepdim=True)
    e = torch.exp(z - m)
    ssum = e.sum(1, keepdim=True)
    p = e / ssum
    a = 1 + (z.abs() + m.abs()) * (z < m)
    pos = torch.arange(H3 * W3, device=y3.device, dtype=torch.float64)
    col, row = (pos % W3).view(1, -1, 1), torch.div(pos, W3, rounding_mode="floor").view(1, -1, 1)
    return z, m, e, ssum, p, a, col, row


def _coords(col, row, control):
    return (row, col) if control == "softargmax_xy_swapped" else (col, row)


# ------------------------------------------------------------------------------------------ forward
def fwd(params, xs_k, y1_k, y2_k, y3_k, feat_k, h4_k, fc, control=None):
    """Forward stages on the kernel's own inputs.  params: the 11 tensors in state_dict order; fc: `fc_paths`.
    Returns {name: (want, scale[, bf16 output])}: y1, y2, y3 NHWC; feat, smax, ssum, h4, emb."""
    W1, b1, W2, b2, W3, b3, temp, W4, b4, W5, b5 = [_d(p) for p in params]
    t = float(temp.reshape(-1)[0])
    res = {}
    v, s = _conv(unpack_xs(xs_k), _w1(control, params[0]), 4, b1)
    res["y1"] = (torch.relu(v).permute(0, 2, 3, 1), s.permute(0, 2, 3, 1), True)
    v, s = _conv(_nchw(y1_k), _conv_w(control, params[2]), 2, b2)
    res["y2"] = (torch.relu(v).permute(0, 2, 3, 1), s.permute(0, 2, 3, 1), True)
    v, s = _conv(_nchw(y2_k), _conv_w(control, params[4]), 1, b3)
    res["y3"] = (torch.relu(v).permute(0, 2, 3, 1), s.permute(0, 2, 3, 1))
    z, m, e, ssum, p, a, col, row = _softmax(y3_k, t)
    cx, cy = _coords(col, row, control)
    N, C = p.shape[0], p.shape[2]
    fx, fy = (p * cx).sum(1), (p * cy).sum(1)
    pa = p * a
    sx = (pa * cx).sum(1) + fx * pa.sum(1)
    sy = (pa * cy).sum(1) + fy * pa.sum(1)
    res["feat"] = (torch.stack([fx, fy], -1).reshape(N, 2 * C), torch.stack([sx, sy], -1).reshape(N, 2 * C))
    res["smax"] = (m.reshape(N, C), m.abs().reshape(N, C))
    res["ssum"] = (ssum.reshape(N, C), (e * a).sum(1))
    o1, o2 = _fc_op(fc["fc1"], control), _fc_op(fc["fc2"], control)
    f = o1(_d(feat_k))
    v, s = f @ o1(W4).t() + b4, f.abs() @ o1(W4).abs().t() + b4.abs()
    res["h4"] = (torch.relu(v), s)
    h = o2(_d(h4_k))
    res["emb"] = (h @ o2(W5).t() + b5, h.abs() @ o2(W5).abs().t() + b5.abs())
    return res


# ------------------------------------------------------------------------------------------ backward
def bwd_workspace(ws, N, H, W, hidden, xs_saved):
    """Views of the backward's intermediates in the workspace after a tacorl_lmp_encoder_bwd call (PREC_BF16), at the
    offsets enc_bwd_tc carves them (Arena: 256-byte granules, in order).  dy3 lives at y2's pitch with a 2-pixel zero
    margin and dy1 at the space-to-depth image's pitch with a 1-pixel zero margin (the linear-shift weight gradients);
    `margins` holds those margins.  xs is there when the backward rebuilt it."""
    H1, W1 = (H - 8) // 4 + 1, (W - 8) // 4 + 1
    H2, W2 = (H1 - 4) // 2 + 1, (W1 - 4) // 2 + 1
    H3, W3 = H2 - 2, W2 - 2
    assert ((128 + W2 + 2 + 7) & ~7) <= 256 and ((128 + W1 + 1 + 15) & ~15) <= 256, "linear-shift layouts expected"
    off = [0]

    def take(nbytes):
        o = off[0]
        off[0] += (nbytes + 255) & ~255
        return ws[o:o + nbytes]

    take(9 * 64 * 64 * 2)
    take(16 * 32 * 64 * 2)
    out = {"dh4": take(N * hidden * 4).view(torch.float32).view(N, hidden),
           "dfeat": take(N * 128 * 4).view(torch.float32).view(N, 128),
           "dtau": take(N * 4).view(torch.float32)}
    take(592 * 64 * 4)
    take(64 << 20)
    dy3 = take(N * H2 * W2 * 64 * 2).view(torch.bfloat16).view(N, H2, W2, 64)
    dy2 = take(N * H2 * W2 * 64 * 2).view(torch.bfloat16).view(N, H2, W2, 64)
    dy1 = take(N * (H1 + 1) * (W1 + 1) * 32 * 2).view(torch.bfloat16).view(N, H1 + 1, W1 + 1, 32)
    out.update(dy3=dy3[:, :H3, :W3], dy2=dy2, dy1=dy1[:, :H1, :W1],
               margins=[dy3[:, H3:], dy3[:, :H3, W3:], dy1[:, H1:], dy1[:, :H1, W1:]])
    if not xs_saved:
        out["xs"] = take(N * (H1 + 1) * (W1 + 1) * 64 * 2).view(torch.bfloat16).view(N, H1 + 1, W1 + 1, 64)
    return out


def _round_mode(control):
    """How the oracle expects the kernels to round dy3 / dy2 / dy1: (want of the fp64 value v, bf16 allowance)."""
    if control == "dy_truncated":
        return (lambda v: (v.float().view(torch.int32) & -65536).view(torch.float32).double()), False
    return (lambda v: v), True


def bwd(params, xs_k, y1_k, y2_k, y3_k, feat_k, h4_k, d_emb, fc, ws_k, pre=None, control=None):
    """Every backward stage on the kernel's own input of that stage.  ws_k: the kernel's intermediates
    (`bwd_workspace`: dh4, dfeat, dy3, dy2, dy1 NHWC; dh4 is ignored on the fused FC head).  pre: the pre-filled
    gradients (accumulate = 1) or None.  Returns {name: (want, scale[, bf16 output])} over PARAMS and dh4 (non-fused
    head only), dfeat, dtau, dy3, dy2, dy1."""
    W1, b1, W2, b2, W3, b3, temp, W4, b4, W5, b5 = [_d(p) for p in params]
    t = float(temp.reshape(-1)[0])
    N = d_emb.shape[0]
    g, feat, h4 = _d(d_emb), _d(feat_k), _d(h4_k)
    fused = fc["dh4"] == "fused"
    res = {}
    # ---- FC head
    ops = {k: _fc_op(fc[k], control) for k in FC_GEMMS}
    a, b = ops["dW5"](g), ops["dW5"](h4)
    res["W5"] = (a.t() @ b, a.abs().t() @ b.abs())
    res["b5"] = (g.sum(0), g.abs().sum(0))
    gate4 = (h4_k > 0).double()
    o = ops["dh4"]
    dh4, sdh4 = (o(g) @ o(W5)) * gate4, (o(g).abs() @ o(W5).abs()) * gate4
    if fused:       # the fused fp32 head keeps dh4 in registers: carry the oracle's value and its scale
        d_in, sd_in = dh4, sdh4
    else:
        res["dh4"] = (dh4, sdh4)
        d_in = _d(ws_k["dh4"])
        sd_in = d_in.abs()
    a, f = ops["dW4"](d_in), ops["dW4"](feat)
    res["W4"] = (a.t() @ f, (sd_in if a is d_in else a.abs()).t() @ f.abs())
    res["b4"] = (d_in.sum(0), sd_in.sum(0))
    a, w4 = ops["dfeat"](d_in), ops["dfeat"](W4)
    res["dfeat"] = (a @ w4, (sd_in if a is d_in else a.abs()) @ w4.abs())
    # ---- soft-argmax backward and temperature, from the kernel's dfeat
    z, m, e, ssum, p, a, col, row = _softmax(y3_k, t)
    cx, cy = _coords(col, row, control)
    C = p.shape[2]
    fk = feat.reshape(N, C, 2)
    fx, fy = fk[..., 0].unsqueeze(1), fk[..., 1].unsqueeze(1)
    dfk = _d(ws_k["dfeat"]).reshape(N, C, 2)
    gx, gy = dfk[..., 0].unsqueeze(1), dfk[..., 1].unsqueeze(1)
    dz = p * (gx * (cx - fx) + gy * (cy - fy))
    sdz = p * (a + (p * a).sum(1, keepdim=True)) * (gx.abs() * (cx + fx.abs()) + gy.abs() * (cy + fy.abs()))
    y3 = _d(y3_k).reshape(N, -1, C)
    dtau, sdtau = -(dz * y3).sum((1, 2)) / t ** 2, (sdz * y3.abs()).sum((1, 2)) / t ** 2
    res["dtau"] = (dtau, sdtau)
    res["temp"] = (dtau.sum().reshape(1), sdtau.sum().reshape(1))
    rnd, half = _round_mode(control)
    gate3 = (y3 > 0).double()
    nhwc = y3_k.shape
    v = (dz * gate3 / t).reshape(nhwc)
    res["dy3"] = (rnd(v), (sdz * gate3 / abs(t)).reshape(nhwc), half)
    # ---- conv stack, each stage from the kernel's own gradient of the stage before
    dy3, dy2, dy1 = (_nchw(ws_k[k]) for k in ("dy3", "dy2", "dy1"))
    y2 = _nchw(y2_k)
    _conv_bwd(res, "W3", "b3", dy3, y2, W3.shape, 1, control, v.permute(0, 3, 1, 2))
    w3 = _conv_w(control, params[4])
    gate2 = (y2 > 0).double() if control != "dy2_no_relu_mask" else torch.ones_like(y2)
    v = conv2d_input(y2.shape, w3, dy3) * gate2
    s = conv2d_input(y2.shape, w3.abs(), dy3.abs()) * gate2
    res["dy2"] = (rnd(v).permute(0, 2, 3, 1), s.permute(0, 2, 3, 1), half)
    y1 = _nchw(y1_k)
    _conv_bwd(res, "W2", "b2", dy2, y1, W2.shape, 2, control, v)
    w2 = _conv_w(control, params[2])
    if control == "conv2_parity_swap":
        w2 = w2.clone()
        w2[:, :, 0::2, 1::2], w2[:, :, 1::2, 0::2] = w2[:, :, 1::2, 0::2].clone(), w2[:, :, 0::2, 1::2].clone()
    gate1 = (y1 > 0).double()
    v = conv2d_input(y1.shape, w2, dy2, stride=2) * gate1
    s = conv2d_input(y1.shape, w2.abs(), dy2.abs(), stride=2) * gate1
    if control == "dy1_scaled":
        v = v * (1 + 2.0 ** -9)
    res["dy1"] = (rnd(v).permute(0, 2, 3, 1), s.permute(0, 2, 3, 1), half)
    x = unpack_xs(xs_k)
    _conv_bwd(res, "W1", "b1", dy1, x, W1.shape, 4, control, v)
    if control == "conv1_taps_transposed":
        res["W1"] = tuple(q.transpose(2, 3) for q in res["W1"])
    if pre is not None and control != "accumulate_ignored":
        for k in PARAMS:
            v, s = res[k]
            q = _d(pre[PARAMS.index(k)])
            res[k] = (v + q, s + q.abs())
    return res


def _conv_bwd(res, wname, bname, dy, x, wshape, stride, control=None, unrounded=None):
    """Weight and bias gradient of one conv from the kernel's bf16 output gradient dy (N, OC, OH, OW).  unrounded: the
    fp64 value dy was rounded from, which the dy_unrounded / bias_from_fp32_dy controls consume instead."""
    dw = unrounded if control == "dy_unrounded" else dy
    db = unrounded if control in ("dy_unrounded", "bias_from_fp32_dy") else dy
    res[wname] = (conv2d_weight(x, wshape, dw, stride=stride), conv2d_weight(x.abs(), wshape, dw.abs(), stride=stride))
    res[bname] = (db.sum((0, 2, 3)), db.abs().sum((0, 2, 3)))


# ------------------------------------------------------------------------------------------ checks
def check(got, want, scale, tau, bf16=False):
    """Per element |got - want| <= tau * scale (+ 1/2 ulp_bf16(want) for bf16 outputs).
    Returns (ok, max excess / scale, index of the worst element): the excess is |got - want| less the half ulp."""
    got = got.detach().to(want.device).double()
    assert got.shape == want.shape, (got.shape, want.shape)
    excess = ((got - want).abs() - (0.5 * ulp_bf16(want) if bf16 else 0)).clamp_min(0)
    ok = bool((excess <= tau * scale + 1e-30).all()) and not bool(got.isnan().any())
    ratio = excess / (scale + 1e-30)
    ratio = torch.where(got.isnan(), torch.full_like(ratio, float("inf")), ratio)
    worst = int(ratio.argmax()) if ratio.numel() else 0
    return ok, float(ratio.max()) if ratio.numel() else 0.0, worst


BF16_OUT = ("y1", "y2", "dy3", "dy2", "dy1")


def check_all(got, ref, tau):
    """got: {name: tensor or None}; ref: {name: (want, scale[, bf16 output])} -> {name: (ok, max ratio)}."""
    return {k: check(got[k], r[0], r[1], tau, len(r) > 2 and r[2])[:2] for k, r in ref.items() if got.get(k) is not None}


def bump_one_ulp(got, want, scale):
    """A copy of bf16 `got` with one element moved by one bf16 ulp away from `want`: the element where a one-ulp error
    is largest against its scale."""
    g = got.detach().clone()
    k = int((want.abs() / (scale + 1e-30)).reshape(-1).argmax())
    flat = g.view(-1)
    v = float(flat[k])
    up = v >= float(want.reshape(-1)[k])
    step = float(ulp_bf16(torch.tensor(v)))
    flat[k] = v + step if up else v - step
    assert float(flat[k]) != v
    return g
