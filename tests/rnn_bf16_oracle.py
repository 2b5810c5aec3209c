"""Teacher-forced fp64 oracle of one direction of the bf16 ReLU-RNN kernels (tacorl_rnn_layer_{fwd,bwd} with
PREC_BF16, tacorl_rnn_layer2_{fwd,bwd}).

A free-running bf16 recurrence feeds its own rounded hidden state back into itself and drifts chaotically away from
fp64 within a few steps.  But every bf16 operand the tensor cores consume is observable: the forward keeps h_t as
fp32 `out` and as its round-to-nearest-even bf16 copy, and the backward overwrites `dout` with the fp32 dpre and
keeps its bf16 copy.  Given the kernel's own bf16 state of the neighbouring step, each step is a fixed function of
bf16-exact operands, and the only error left is the kernel's fp32 accumulation.  So every formula here takes the
kernel's tensors (marked K) as inputs and is checked per element against `scale`, the same contraction run on
absolute values, at a tolerance near fp32 rounding.  Every step's inputs are known up front, so each formula is a
few large fp64 products over all steps at once, not a sequential loop.

Tensors are time-major (T, B, features) views of ONE direction, any dtype and device; results are float64.  Only the
active steps take part: forward t = 0 .. n-1, reverse t = T-n .. T-1 (run from T-1 down).

`control` alters the oracle the way a subtle kernel bug would (the tests assert that the check then fails):
  "fp32_hidden"  the unrounded fp32 hidden state instead of its bf16 copy;
  "shift_pairs"  dW_hh pairs dpre[t] with h[t] instead of h[prev(t)];
  "drop_h0"      dW_hh without the dpre[first]^T h0 term;
  "ignore_dhn"   the gradient arriving at the last hidden state is dropped.
"""
import torch

CONTROLS = ("fp32_hidden", "shift_pairs", "drop_h0", "ignore_dhn")
# per-element bar |got - want| <= TAU * scale (calibration: tests/test_gpu_rnn_bf16_oracle.py)
TAU = 1e-5


def rne(t):
    """The bf16 value the kernels feed the tensor cores (round to nearest even), as float64."""
    return t.float().bfloat16().double()


def _d(t):
    return None if t is None else t.double()


def active(T, n, reverse):
    """Active steps as a slice of the time axis (ascending t)."""
    return slice(T - n, T) if reverse else slice(0, n)


def _hidden(out_k, control):
    return out_k.double() if control == "fp32_hidden" else rne(out_k)


def _h_prev(out_k, h0, n, reverse, control=None):
    """(n, B, H): the bf16 hidden state each active step consumes (h0 or 0 for the first one), ascending t."""
    T, B, H = out_k.shape
    hb = _hidden(out_k, control)
    first = rne(h0).unsqueeze(0) if h0 is not None else hb.new_zeros(1, B, H)
    if reverse:
        return torch.cat([hb[T - n + 1:T], first], 0)
    return torch.cat([first, hb[0:n - 1]], 0)


def _mm(a, b):
    """(value, scale) of a @ b."""
    return a @ b, a.abs() @ b.abs()


def _flat(t):
    return t.reshape(-1, t.shape[-1])


def fwd(x, w_ih, w_hh, b_ih, b_hh, out_k, h0=None, reverse=False, n=None, control=None):
    """h[t] = relu(rne(x[t]) rne(W_ih)^T + b_ih + b_hh + hb[prev(t)] rne(W_hh)^T) over the active steps.
    out_k (K): the kernel's fp32 hidden states (T, B, H).  Returns {"out": (want, scale)}, (n, B, H)."""
    T = x.shape[0]
    n = T if n is None else n
    a = active(T, n, reverse)
    xin, xs = _mm(rne(x[a]), rne(w_ih).t())
    hin, hs = _mm(_h_prev(out_k, h0, n, reverse, control), rne(w_hh).t())
    bias = _d(b_ih) + _d(b_hh)
    return {"out": (torch.relu(xin + bias + hin), xs + bias.abs() + hs)}


def bwd(x, w_ih, w_hh, out_k, dout_in, dpre_k, h0=None, dhn=None, reverse=False, n=None, control=None):
    """BPTT of one direction, teacher-forced on the kernel's dpre.
      out_k (K): fp32 hidden states; dout_in: dL/dout as passed in; dpre_k (K): the `dout` buffer after the call.
    Returns {name: (want, scale)}: dpre (n,B,H) over the active steps, dw_ih, dw_hh, db (the fp32 column sum of
    dpre_k: db_ih == db_hh), dx (n,B,I) over the active steps, dh0 (B,H).  Pre-filled (accumulated) outputs and rows
    outside the active range are the caller's to add."""
    T, B, H = out_k.shape
    n = T if n is None else n
    a = active(T, n, reverse)
    gate = (out_k[a] > 0).double()
    db = rne(dpre_k[a])
    whh = rne(w_hh)
    # gradient carried into each active step from the next step of the chain (t + 1 forward, t - 1 reverse)
    carry, carry_s = _mm(db, whh)
    z = carry.new_zeros(1, B, H)
    last = dhn.double().unsqueeze(0) if (dhn is not None and control != "ignore_dhn") else z
    if reverse:
        carry, carry_s = torch.cat([last, carry[:-1]], 0), torch.cat([last.abs(), carry_s[:-1]], 0)
    else:
        carry, carry_s = torch.cat([carry[1:], last], 0), torch.cat([carry_s[1:], last.abs()], 0)
    d_in = dout_in[a].double()
    res = {"dpre": ((d_in + carry) * gate, (d_in.abs() + carry_s) * gate)}
    hp = _h_prev(out_k, h0 if control != "drop_h0" else None, n, reverse, control)
    if control == "shift_pairs":      # dpre[t] with h[t]: the pairing one step off
        hb = rne(out_k[a])
        hp = torch.cat([hb[:-1], hp[-1:]], 0) if reverse else torch.cat([hp[:1], hb[1:]], 0)
    res["dw_hh"] = _mm(_flat(db).t(), _flat(hp))
    res["dw_ih"] = _mm(_flat(db).t(), _flat(rne(x[a])))
    dp = _flat(dpre_k[a].double())
    res["db"] = (dp.sum(0), dp.abs().sum(0))
    res["dx"] = _mm(db, rne(w_ih))
    first = db[-1] if reverse else db[0]
    res["dh0"] = _mm(first, whh)
    return res


def check(got, want, scale, tau):
    """Per-element |got - want| <= tau * scale + 1e-30.  Returns (ok, max |got - want| / scale, per-step relative L2
    errors along the leading axis, index of the worst element)."""
    got = got.detach().to(want.device).double()
    assert got.shape == want.shape, (got.shape, want.shape)
    err = (got - want).abs()
    ok = bool((err <= tau * scale + 1e-30).all())
    ratio = err / (scale + 1e-30)
    worst = int(ratio.argmax()) if ratio.numel() else 0
    if want.dim() >= 2:
        steps = ((got - want).flatten(1).norm(dim=1) / (want.flatten(1).norm(dim=1) + 1e-30)).tolist()
    else:
        steps = [float((got - want).norm() / (want.norm() + 1e-30))]
    return ok, float(ratio.max()) if ratio.numel() else 0.0, steps, worst


def check_all(got, ref, tau):
    """got: {name: tensor or None}; ref: {name: (want, scale)} -> {name: (ok, max ratio, per-step errors)} over the
    names present in both."""
    return {k: check(got[k], *ref[k], tau)[:3] for k in ref if got.get(k) is not None}


def bump_one_ulp(got, want, scale):
    """A copy of `got` with one element moved up by one bf16 ulp of its value: the element where a one-ulp error is
    largest against its scale."""
    g = got.detach().clone()
    k = int((want.abs() / (scale + 1e-30)).argmax())
    flat = g.view(-1)
    v = float(flat[k])
    e = torch.frexp(torch.tensor(abs(v) if v != 0 else 1.0, dtype=torch.float64))[1].item()
    flat[k] = v + 2.0 ** (e - 1 - 7)     # bf16 keeps 8 significant bits: ulp = 2^(exponent - 7)
    return g
