"""torch.autograd.Function wrappers over the C-ABI kernels (include/tacorl_b200.h).

PyTorch is used for device memory, streams and autograd bookkeeping only; every
contraction / reduction / loss below runs in libtacorl_b200.so.  No CPU path exists.
"""
import ctypes
import math
import weakref

import torch
from torch.autograd import Function

from . import _lib as L

_STATE = {"prec": L.PREC_F32}
_GEMM_WS = 96 << 20


def set_precision(name):
    """'fp32' = full-fp32 SIMT parity path; 'bf16' = bf16 tcgen05 operands, fp32 accumulate."""
    _STATE["prec"] = {"fp32": L.PREC_F32, "bf16": L.PREC_BF16}[name]


def get_precision():
    return "bf16" if _STATE["prec"] == L.PREC_BF16 else "fp32"


_SIDE = {}


def _side_stream(dev):
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=dev)
    return _SIDE[key]


def _prep_stream(dev):
    key = ("prep", dev.index if dev.index is not None else torch.cuda.current_device())
    if key not in _SIDE:
        _SIDE[key] = torch.cuda.Stream(device=dev)
    return _SIDE[key]


def _off(t, elems):
    return ctypes.c_void_p(t.data_ptr() + 4 * elems)


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


def _ld(t):
    assert t.dim() == 2 and (t.stride(1) == 1 or t.shape[1] == 1), "row-major 2-D view expected"
    return t.stride(0) if t.shape[0] > 1 else max(t.shape[1], t.stride(0))


# ---- bf16 shadow copies of optimiser-owned parameters.  tacorl_b200.optim.FlatAdam keeps a bf16 twin of its flat fp32
# parameter buffer (written by the Adam kernel itself); the tensor-core ops read weights from it instead of casting the
# fp32 weights on every call.  A parameter's slice of the twin is (re)cast lazily when the parameter's or the flat
# buffer's torch version counter moved (load_state_dict, broadcast, manual init): raw kernel writes do not bump them.
_SHADOW_OWNERS = weakref.WeakSet()      # optimisers come and go (tests, re-configured modules): no strong references


def register_shadow_owner(owner):
    """owner: object with .pbuf.flat (fp32), .shadow (bf16, same numel), ._pver (dict) and ._flat_version."""
    _SHADOW_OWNERS.add(owner)


def refresh_shadows():
    """Re-validate every registered parameter (used before replaying a captured step)."""
    for o in list(_SHADOW_OWNERS):
        for p in o.param_groups[0]["params"]:
            shadow_of(p)
    for key, (ref, ver, sh) in list(_FROZEN_SHADOWS.items()):
        t = ref()
        if t is None or t.data_ptr() != key or t.requires_grad:
            del _FROZEN_SHADOWS[key]
        elif t._version != ver:
            with torch.no_grad():
                sh.copy_(t.detach().reshape(-1))          # in place: captured graphs keep reading the same address
            _FROZEN_SHADOWS[key] = (ref, t._version, sh)


# bf16 twins of FROZEN parameters: modules registered with mark_frozen() (TACO-RL's frozen plan recogniser, tacorl.py:
# 124-125), requires_grad False, owned by no optimiser.  Cast once and re-cast when the tensor's torch version counter
# moves (load_state_dict, copy_).  Only registered parameters qualify: nothing that a kernel updates through raw
# pointers (Polyak targets) may be cached, a captured graph would never see the refresh.
_FROZEN_SHADOWS = {}
_FROZEN_PARAMS = {}                 # id(parameter) -> weakref


def mark_frozen(module):
    """Declare every parameter of `module` frozen for good (the caller also sets requires_grad False)."""
    for p in module.parameters():
        _FROZEN_PARAMS[id(p)] = weakref.ref(p)


def invalidate_frozen_shadows():
    _FROZEN_SHADOWS.clear()


def _frozen_shadow_of(t):
    ref = _FROZEN_PARAMS.get(id(t))
    if ref is None or ref() is not t or t.requires_grad or t.dtype != torch.float32:
        return None
    key = t.data_ptr()
    hit = _FROZEN_SHADOWS.get(key)
    if hit is not None:
        ref, ver, sh = hit
        if ref() is t and sh.numel() == t.numel():
            if ver != t._version:
                with torch.no_grad():
                    sh.copy_(t.detach().reshape(-1))
                _FROZEN_SHADOWS[key] = (ref, t._version, sh)
            return sh
    if torch.cuda.is_current_stream_capturing():
        return None                                   # (never allocate a long-lived buffer from a graph's private pool)
    with torch.no_grad():
        sh = t.detach().reshape(-1).to(torch.bfloat16)
    _FROZEN_SHADOWS[key] = (weakref.ref(t), t._version, sh)
    return sh


def shadow_of(t):
    """bf16 twin (flat view) of a whole fp32 parameter that lives inside a registered flat buffer, else None."""
    if _STATE["prec"] != L.PREC_BF16 or t is None or not t.is_cuda or not t.is_contiguous():
        return None
    ptr = t.data_ptr()
    for o in list(_SHADOW_OWNERS):
        flat = o.pbuf.flat
        base = flat.data_ptr()
        if base <= ptr < base + flat.numel() * 4 and flat.device == t.device:
            n = o._pnumel.get(ptr)
            if n != t.numel():
                return None                       # not a whole registered parameter
            if o._flat_version != flat._version:  # the flat buffer itself was edited (e.g. broadcast): all stale
                o._pver.clear()
                o._flat_version = flat._version
            off = (ptr - base) // 4
            sh = o.shadow[off:off + n]
            if o._pver.get(ptr) != t._version:
                with torch.no_grad():
                    sh.copy_(t.detach().reshape(-1))
                o._pver[ptr] = t._version
            return sh
    return _frozen_shadow_of(t)


# ---- gradient slots.  FlatAdam owns one flat gradient buffer; a backward kernel that produces the whole gradient of a
# registered parameter can write it straight into that parameter's slice (and hand autograd the view) instead of into
# a temporary that step() would then copy (189 MB read + write per PlayLMP step).  A slot is handed out at most once
# between two step()/zero_grad() calls, and only while the owning parameter's .grad is None: a second backward through
# the same weight (shared weight, gradient accumulation, zero_grad(set_to_none=False), no zero_grad at all) gets a
# temporary, and autograd accumulates it into the existing .grad as usual -- never a kernel write over a live .grad.
_GRAD_OWNERS = weakref.WeakSet()


def register_grad_owner(owner):
    """owner: object with .pbuf.flat, .flat_grad (same numel), ._pnumel (data_ptr -> numel), ._pparam (data_ptr ->
    parameter) and ._slots_taken (set)."""
    _GRAD_OWNERS.add(owner)


def grad_slot_of(t):
    """View of the owning optimiser's flat gradient for the whole parameter `t` (first request since the last
    step()/zero_grad()), else None."""
    if t is None or not t.is_cuda or not t.is_contiguous():
        return None
    ptr = t.data_ptr()
    for o in list(_GRAD_OWNERS):
        flat = o.pbuf.flat
        base = flat.data_ptr()
        if base <= ptr < base + flat.numel() * 4 and flat.device == t.device:
            if o._pnumel.get(ptr) != t.numel() or ptr in o._slots_taken:
                return None
            owner_param = o._pparam.get(ptr)
            if owner_param is None or owner_param.grad is not None:
                return None
            o._slots_taken.add(ptr)
            off = (ptr - base) // 4
            return o.flat_grad[off:off + t.numel()].view(t.shape)
    return None


def gemm(A, B, C, transA=False, transB=False, alpha=1.0, beta=0.0, bias=None, act=L.ACT_NONE, Cpre=None, A_bf16=None,
         B_bf16=None):
    """C = act(alpha * op(A) op(B) + beta*C + bias); A, B, C are row-major 2-D (possibly strided rows).
    A_bf16 / B_bf16: optional dense bf16 copies of A / B (see shadow_of)."""
    M, N = C.shape
    K = A.shape[0] if transA else A.shape[1]
    assert (A.shape[1] if transA else A.shape[0]) == M, (A.shape, C.shape, transA)
    assert (B.shape[0] if transB else B.shape[1]) == N and (B.shape[1] if transB else B.shape[0]) == K
    ws = L.workspace(_GEMM_WS, C.device)
    L.call("tacorl_gemm_ex", int(transA), int(transB), M, N, K, float(alpha), L.ptr(A), _ld(A), L.ptr(B), _ld(B),
           float(beta), L.ptr(C), _ld(C), L.ptr(bias), int(act), L.ptr(Cpre), _ld(Cpre) if Cpre is not None else 0,
           L.ptr_any(A_bf16), L.ptr_any(B_bf16), ctypes.c_void_p(ws.data_ptr()), ws.numel(),
           _STATE["prec"], L.stream())
    return C


def colsum(X, out=None, accumulate=False):
    M, N = X.shape
    if out is None:
        out = torch.empty(N, device=X.device, dtype=torch.float32)
    L.call("tacorl_colsum", M, N, L.ptr(X), _ld(X), L.ptr(out), int(accumulate), L.stream())
    return out


def scale(x, dev_scalar=None, c=1.0, out=None):
    x = _c(x)
    if out is None:
        out = torch.empty_like(x)
    L.call("tacorl_scale", x.numel(), L.ptr(x), L.ptr(dev_scalar), float(c), L.ptr(out), L.stream())
    return out


# --------------------------------------------------------------------------------------- linear
class LinearFn(Function):
    @staticmethod
    def forward(ctx, x, W, b, act):
        K = W.shape[1]
        x2 = _c(x.reshape(-1, K))
        Wc = _c(W)
        out = torch.empty(x2.shape[0], W.shape[0], device=x.device, dtype=torch.float32)
        pre = torch.empty_like(out) if act == L.ACT_SILU else None
        gemm(x2, Wc, out, transB=True, bias=b, act=act, Cpre=pre, B_bf16=shadow_of(Wc))
        ctx.act = act
        ctx.has_bias = b is not None
        ctx.xshape = x.shape
        ctx.save_for_backward(x2, Wc, pre if act == L.ACT_SILU else (out if act == L.ACT_RELU else None))
        return out.view(*x.shape[:-1], W.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, W, saved = ctx.saved_tensors
        N = W.shape[0]
        dz = _c(dy.reshape(-1, N))
        if ctx.act != L.ACT_NONE:
            dz2 = torch.empty_like(dz)
            L.call("tacorl_act_bwd", ctx.act, dz.numel(), L.ptr(dz), L.ptr(saved), L.ptr(dz2), L.stream())
            dz = dz2
        dx = dW = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x2)
            gemm(dz, W, dx, B_bf16=shadow_of(W))
            dx = dx.view(ctx.xshape)
        if ctx.needs_input_grad[1]:
            dW = torch.empty_like(W)
            gemm(dz, x2, dW, transA=True)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = colsum(dz)
        return dx, dW, db, None


def linear(x, W, b=None, act=None):
    return LinearFn.apply(x, W, b, L.ACTS[act] if not isinstance(act, int) else act)


# --------------------------------------------------------------------------------------- fused MLP chains
def _dp(t):
    return None if t is None else t.data_ptr()


class MlpChainFn(Function):
    """Linear -> act -> ... -> Linear in one launch each way (tacorl_mlp_chain_{fwd,bwd}).
    spec = (acts, segs): acts[l] for the hidden layers; segs[l] = number of (W, b) pairs stacked in layer l (1..3).
    params: per layer, per segment: W, b."""

    @staticmethod
    def _layers(spec, params, in0, grads=None):
        acts, segs = spec
        arr = (L.MlpLayer * len(segs))()
        i, width = 0, in0
        for l, ns in enumerate(segs):
            e = arr[l]
            for sg in range(ns):
                W, b = params[i + 2 * sg], params[i + 2 * sg + 1]
                setattr(e, f"W{sg}", _dp(W)); setattr(e, f"b{sg}", _dp(b)); setattr(e, f"n{sg}", W.shape[0])
                if grads is not None:
                    setattr(e, f"dW{sg}", _dp(grads[i + 2 * sg])); setattr(e, f"db{sg}", _dp(grads[i + 2 * sg + 1]))
            e.in_ = width
            e.act = acts[l] if l < len(acts) else L.ACT_NONE
            width = e.n0 + e.n1 + e.n2
            i += 2 * ns
        return arr, width

    @staticmethod
    def forward(ctx, spec, x0, x1, *params):
        lead = x0.shape[:-1]
        x0 = _c(x0.reshape(-1, x0.shape[-1]))
        x1 = _c(x1.reshape(-1, x1.shape[-1])) if x1 is not None else None
        params = [None if p is None else _c(p) for p in params]
        rows = x0.shape[0]
        in0 = x0.shape[1] + (x1.shape[1] if x1 is not None else 0)
        arr, out_w = MlpChainFn._layers(spec, params, in0)
        nl = len(spec[1])
        zw = sum(arr[l].n0 + arr[l].n1 + arr[l].n2 for l in range(nl - 1))
        z = torch.empty(rows, max(zw, 1), device=x0.device, dtype=torch.float32)
        out = torch.empty(rows, out_w, device=x0.device, dtype=torch.float32)
        L.call("tacorl_mlp_chain_fwd", nl, rows, ctypes.byref(arr), L.ptr(x0), x0.shape[1], x0.shape[1],
               L.ptr(x1), x1.shape[1] if x1 is not None else 0, x1.shape[1] if x1 is not None else 0,
               L.ptr(z), z.shape[1], L.ptr(out), out_w, L.stream())
        ctx.spec, ctx.lead, ctx.has_x1 = spec, lead, x1 is not None
        ctx.save_for_backward(x0, x1, z, *params)
        return out.view(*lead, out_w)

    @staticmethod
    def backward(ctx, d_out):
        x0, x1, z, *params = ctx.saved_tensors
        rows = x0.shape[0]
        d_out = _c(d_out.reshape(rows, -1))
        need = ctx.needs_input_grad
        # a layer's weights either all receive a gradient or none does (detached parameters: input gradient only)
        want_w = any(need[3:])
        grads = [torch.empty_like(p) if (want_w and p is not None) else None for p in params]
        in0 = x0.shape[1] + (x1.shape[1] if x1 is not None else 0)
        arr, _ = MlpChainFn._layers(ctx.spec, params, in0, grads)
        dx0 = torch.empty_like(x0) if need[1] else None
        dx1 = torch.empty_like(x1) if (x1 is not None and need[2]) else None
        nl = len(ctx.spec[1])
        nbytes = L.query("tacorl_mlp_chain_ws_bytes", nl, rows, ctypes.byref(arr))
        ws = L.workspace(nbytes, x0.device, "mlp_chain")
        L.call("tacorl_mlp_chain_bwd", nl, rows, ctypes.byref(arr), L.ptr(x0), x0.shape[1], x0.shape[1],
               L.ptr(x1), x1.shape[1] if x1 is not None else 0, x1.shape[1] if x1 is not None else 0,
               L.ptr(z), z.shape[1], L.ptr(d_out), d_out.shape[1], L.ptr(dx0), x0.shape[1],
               L.ptr(dx1), x1.shape[1] if x1 is not None else 0, ctypes.c_void_p(ws.data_ptr()), ws.numel(), L.stream())
        gx0 = dx0.view(*ctx.lead, x0.shape[1]) if dx0 is not None else None
        gx1 = dx1.view(*ctx.lead, x1.shape[1]) if dx1 is not None else None
        return (None, gx0, gx1, *[g if need[3 + i] else None for i, g in enumerate(grads)])


def mlp_chain(xs, layers, acts):
    """y = Linear_L(... act_1(Linear_1(cat(xs))) ...) in one fused launch (fp32; tacorl_mlp_chain_fwd/bwd).
    xs: one tensor or a pair concatenated along the last dim; layers: per layer a (W, b) pair or a list of up to three pairs
    stacked along the output dim; acts: activation names of the hidden layers (len(layers) - 1 entries).
    Shapes outside the kernel's range (widths > 256 or not multiples of 4, > 4 layers, > 256 rows) run layer by layer."""
    xs = list(xs) if isinstance(xs, (list, tuple)) else [xs]
    segs = [[l] if torch.is_tensor(l[0]) else list(l) for l in layers]
    acts_i = tuple(L.ACTS[a] if not isinstance(a, int) else a for a in acts)
    in0 = sum(x.shape[-1] for x in xs)
    widths = [in0] + [sum(W.shape[0] for W, _ in sg) for sg in segs]
    ok = (len(segs) <= 4 and len(xs) <= 2 and all(len(sg) <= 3 for sg in segs) and xs[0].is_cuda
          and all(w % 4 == 0 and w <= 256 for w in widths[:-1]) and widths[-1] <= 256
          and all(x.dtype == torch.float32 for x in xs) and xs[0].numel() // xs[0].shape[-1] <= 256)
    if not ok:
        x = xs[0] if len(xs) == 1 else torch.cat(xs, dim=-1)
        for l, sg in enumerate(segs):
            W = sg[0][0] if len(sg) == 1 else torch.cat([w for w, _ in sg], dim=0)
            b = sg[0][1] if len(sg) == 1 else torch.cat([bb for _, bb in sg], dim=0)
            x = linear(x, W, b, acts_i[l] if l < len(acts_i) else None)
        return x
    flat = []
    for sg in segs:
        for W, b in sg:
            flat += [W, b]
    spec = (acts_i, tuple(len(sg) for sg in segs))
    return MlpChainFn.apply(spec, xs[0], xs[1] if len(xs) == 2 else None, *flat)


# --------------------------------------------------------------------------------------- encoder
class LMPEncoderFn(Function):
    """LMPVisionEncoder forward/backward as one op (tacorl_lmp_encoder_{fwd,bwd})."""

    @staticmethod
    def forward(ctx, x, save, norm, *params):
        N, C, H, W = x.shape
        assert C == 3, "LMPVisionEncoder kernels are built for 3 input channels"
        if (not x.is_contiguous() and x.dtype == torch.uint8 and x.stride(-1) == 1 and W % 4 == 0
                and all(st % 4 == 0 for st in x.stride()[:-1]) and x.storage_offset() % 4 == 0):
            # strided frame selections (window[:, 0], window[:, -1]): torch's byte-wise strided copy runs at ~0.4 TB/s
            xc = torch.empty(x.shape, device=x.device, dtype=torch.uint8)
            xc.view(torch.int32).copy_(x.view(torch.int32))
            x = xc
        x = _c(x)
        if x.dtype == torch.uint8:       # raw frames: (u8/255 - mean)/std fused into the first kernel
            mean, std = norm
            ctx.xnorm = (1, 1.0 / (255.0 * std), -mean / std)
        else:
            assert x.dtype == torch.float32, f"images must be float32 or uint8, got {x.dtype}"
            ctx.xnorm = (0, 1.0, 0.0)
        params = [_c(p) for p in params]
        hidden, latent = params[7].shape[0], params[9].shape[0]
        dev = x.device
        H1, W1 = (H - 8) // 4 + 1, (W - 8) // 4 + 1
        H2, W2 = (H1 - 4) // 2 + 1, (W1 - 4) // 2 + 1
        H3, W3 = H2 - 2, W2 - 2
        emb = torch.empty(N, latent, device=dev, dtype=torch.float32)
        if save:
            adt = torch.bfloat16 if _STATE["prec"] == L.PREC_BF16 else torch.float32
            y1 = torch.empty(N, H1, W1, 32, device=dev, dtype=adt)
            y2 = torch.empty(N, H2, W2, 64, device=dev, dtype=adt)
            y3 = torch.empty(N, H3, W3, 64, device=dev)
            feat = torch.empty(N, 128, device=dev)
            smax = torch.empty(N, 64, device=dev)
            ssum = torch.empty(N, 64, device=dev)
            h4 = torch.empty(N, hidden, device=dev)
            # bf16 path: keep conv1's space-to-depth input so the backward pass does not rebuild it from the frames
            xs = (torch.empty(N, H1 + 1, W1 + 1, 64, device=dev, dtype=torch.bfloat16)
                  if _STATE["prec"] == L.PREC_BF16 else None)
        else:
            y1 = y2 = y3 = feat = smax = ssum = h4 = xs = None
        nbytes = L.query("tacorl_lmp_encoder_ws_bytes", N, H, W, hidden, latent, 0)
        ws = L.workspace(nbytes, dev)
        ctx.prec = _STATE["prec"]
        L.call("tacorl_lmp_encoder_fwd", L.ptr_any(x), *ctx.xnorm, N, H, W, L.ptr_array(params), hidden, latent, L.ptr_any(y1),
               L.ptr_any(y2), L.ptr(y3), L.ptr(feat), L.ptr(smax), L.ptr(ssum), L.ptr(h4), L.ptr(emb), L.ptr_any(xs),
               ctypes.c_void_p(ws.data_ptr()), ws.numel(), _STATE["prec"], L.stream())
        if save:
            ctx.has_xs = xs is not None
            ctx.save_for_backward(x, y1, y2, y3, feat, smax, ssum, h4, *((xs,) if xs is not None else ()), *params)
        ctx.dims = (N, H, W, hidden, latent)
        return emb

    @staticmethod
    def backward(ctx, d_emb):
        x, y1, y2, y3, feat, smax, ssum, h4, *params = ctx.saved_tensors
        xs = params.pop(0) if ctx.has_xs else None
        N, H, W, hidden, latent = ctx.dims
        grads = [torch.empty_like(p) for p in params]
        nbytes = L.query("tacorl_lmp_encoder_ws_bytes", N, H, W, hidden, latent, 1)
        ws = L.workspace(nbytes, x.device)
        d_emb = _c(d_emb)
        L.call("tacorl_lmp_encoder_bwd", L.ptr_any(x), *ctx.xnorm, N, H, W, L.ptr_array(params), hidden, latent, L.ptr_any(y1),
               L.ptr_any(y2), L.ptr(y3), L.ptr(feat), L.ptr(smax), L.ptr(ssum), L.ptr(h4), L.ptr(d_emb),
               L.ptr_array(grads), 0, L.ptr_any(xs), ctypes.c_void_p(ws.data_ptr()), ws.numel(), ctx.prec, L.stream())
        return (None, None, None, *grads)


def lmp_encoder(x, params, norm=(0.5, 0.5)):
    """params: the 11 tensors in state_dict order.  Images never receive a gradient.
    x: float32 (N,3,H,W) already normalised, or uint8 raw frames normalised on the device with norm=(mean, std)."""
    save = torch.is_grad_enabled() and any(p.requires_grad for p in params)
    return LMPEncoderFn.apply(x, save, norm, *params)


# --------------------------------------------------------------------------------------- RNN
class ReluRNNFn(Function):
    """Multi-layer (bi)directional ReLU RNN on time-major input (T,B,I).
    weights: per layer, per direction: w_ih, w_hh, b_ih, b_hh (torch nn.RNN order).
    last_only: return only out[T-1] (B, D*H); the top layer's reverse direction then runs one step."""

    @staticmethod
    def forward(ctx, x, h0, num_layers, bidir, last_only, *weights):
        T, B, I = x.shape
        D = 2 if bidir else 1
        H = weights[1].shape[0]
        x = _c(x)
        weights = [_c(w) for w in weights]
        dev = x.device
        outs = []
        inp = x
        hn = [] if not last_only else None
        # bf16 training: keep the bf16 hidden states for BPTT, and transpose W_hh (the carry GEMM's operand) on the
        # side stream now, where it overlaps the latency-bound recurrence, instead of on the backward's critical path
        train = _STATE["prec"] == L.PREC_BF16 and any(ctx.needs_input_grad)   # (grad mode itself is off inside forward)
        hbs = [torch.empty(T, B, H, device=dev, dtype=torch.bfloat16) if train else None for _ in range(num_layers * D)]
        whts, prep_done = [None] * (num_layers * D), None
        if train:
            main, prep = torch.cuda.current_stream(dev), _prep_stream(dev)
            whts = [torch.empty(H, H, device=dev, dtype=torch.bfloat16) for _ in range(num_layers * D)]   # main-stream pool
            prep.wait_stream(main)
            with torch.cuda.stream(prep):
                for k in range(num_layers * D):
                    L.call("tacorl_cast_transpose_bf16", L.ptr(weights[k * 4 + 1]), H, H, L.ptr_any(whts[k]), L.stream())
                prep_done = torch.cuda.Event()
                prep_done.record(prep)
        for l in range(num_layers):
            Il = inp.shape[2]
            out = torch.empty(T, B, D * H, device=dev, dtype=torch.float32)
            nbytes = L.query("tacorl_rnn_layer_ws_bytes", T, B, Il, H)

            def run_dir(d, tag):
                w_ih, w_hh, b_ih, b_hh = weights[(l * D + d) * 4:(l * D + d) * 4 + 4]
                n_steps = 1 if (last_only and l == num_layers - 1 and d == 1) else T
                h0_ld = None if h0 is None else _c(h0[l * D + d])
                ws = L.workspace(nbytes, dev, tag)
                L.call("tacorl_rnn_layer_fwd", T, B, Il, H, L.ptr(inp), Il, L.ptr(w_ih), L.ptr(w_hh), L.ptr(b_ih),
                       L.ptr(b_hh), L.ptr(h0_ld), d, n_steps, _off(out, d * H), D * H,
                       L.ptr_any(shadow_of(w_ih)), L.ptr_any(shadow_of(w_hh)), L.ptr_any(hbs[l * D + d]),
                       ctypes.c_void_p(ws.data_ptr()), ws.numel(), _STATE["prec"], L.stream())

            if D == 2:
                # the two directions of a layer are independent: the reverse one runs on a side stream
                # (own workspace), joined before the next layer reads the concatenated output.  Step-by-step
                # launches here: two persistent launches would be chained one after the other (they may never
                # be co-scheduled), which measured slower than letting the per-step kernels of the two
                # directions interleave (BiRNN fwd+bwd 1.16 ms vs 1.12 ms).
                main, side = torch.cuda.current_stream(dev), _side_stream(dev)
                side.wait_stream(main)
                was = L.lib().tacorl_rnn_seq_enable(0)
                try:
                    with torch.cuda.stream(side):
                        run_dir(1, "rnn_side")
                    run_dir(0, "main")
                finally:
                    L.lib().tacorl_rnn_seq_enable(was)
                main.wait_stream(side)
            else:
                run_dir(0, "main")
            if hn is not None:
                for d in range(D):
                    hn.append(out[0 if d == 1 else T - 1, :, d * H:(d + 1) * H])
            outs.append(out)
            inp = out
        ctx.cfg = (T, B, I, H, D, num_layers, last_only)
        ctx.has_h0 = h0 is not None
        ctx.bf16_aux = (hbs, whts, prep_done) if train else None
        ctx.save_for_backward(x, h0, *outs, *weights)
        if last_only:
            return inp[T - 1], None
        return inp, torch.stack(hn, dim=0)

    @staticmethod
    def backward(ctx, d_out, d_hn):
        T, B, I, H, D, num_layers, last_only = ctx.cfg
        saved = ctx.saved_tensors
        x, h0 = saved[0], saved[1]
        outs = saved[2:2 + num_layers]
        weights = saved[2 + num_layers:]
        dev = x.device
        if last_only:
            dbuf = torch.zeros(T, B, D * H, device=dev, dtype=torch.float32)
            dbuf[T - 1].copy_(d_out)
        else:
            dbuf = d_out.contiguous().clone() if d_out is not None else torch.zeros(T, B, D * H, device=dev)
        wgrads = [None] * len(weights)
        dh0 = torch.empty_like(h0) if (ctx.has_h0 and ctx.needs_input_grad[1]) else None
        aux = ctx.bf16_aux if _STATE["prec"] == L.PREC_BF16 else None
        hbs, whts = (aux[0], aux[1]) if aux is not None else ([None] * (num_layers * D),) * 2
        if aux is not None:
            torch.cuda.current_stream(dev).wait_event(aux[2])
        for l in range(num_layers - 1, -1, -1):
            inp = x if l == 0 else outs[l - 1]
            Il = inp.shape[2]
            need_dx = l > 0 or ctx.needs_input_grad[0]
            dx = torch.empty(T, B, Il, device=dev, dtype=torch.float32) if need_dx else None
            dx_rev = torch.empty(T, B, Il, device=dev, dtype=torch.float32) if (need_dx and D == 2) else None
            nbytes = L.query("tacorl_rnn_layer_ws_bytes", T, B, Il, H)

            def run_dir(d, tag, dx_buf):
                k = (l * D + d) * 4
                w_ih, w_hh = weights[k], weights[k + 1]
                g = []
                for j in range(4):     # straight into the optimiser's flat gradient when this is the parameter's first use
                    slot = grad_slot_of(weights[k + j])
                    g.append(slot if slot is not None else torch.empty_like(weights[k + j]))
                n_steps = 1 if (last_only and l == num_layers - 1 and d == 1) else T
                h0_ld = None if h0 is None else _c(h0[l * D + d])
                dhn_ld = None if d_hn is None else _c(d_hn[l * D + d])
                dh0_ld = None if dh0 is None else dh0[l * D + d]
                ws = L.workspace(nbytes, dev, tag)
                L.call("tacorl_rnn_layer_bwd", T, B, Il, H, L.ptr(inp), Il, L.ptr(w_ih), L.ptr(w_hh), L.ptr(h0_ld),
                       d, n_steps, _off(outs[l], d * H), D * H, _off(dbuf, d * H), D * H, L.ptr(dhn_ld),
                       L.ptr(dx_buf), Il, 0, L.ptr(g[0]), L.ptr(g[1]), L.ptr(g[2]), L.ptr(g[3]), 0,
                       L.ptr(dh0_ld), L.ptr_any(shadow_of(w_ih)), L.ptr_any(whts[l * D + d]), L.ptr_any(hbs[l * D + d]),
                       ctypes.c_void_p(ws.data_ptr()), ws.numel(), _STATE["prec"], L.stream())
                wgrads[k:k + 4] = g

            if D == 2:
                main, side = torch.cuda.current_stream(dev), _side_stream(dev)
                side.wait_stream(main)
                was = L.lib().tacorl_rnn_seq_enable(0)
                try:
                    with torch.cuda.stream(side):
                        run_dir(1, "rnn_side", dx_rev)
                    run_dir(0, "main", dx)
                finally:
                    L.lib().tacorl_rnn_seq_enable(was)
                main.wait_stream(side)
                if need_dx:
                    dx.add_(dx_rev)
            else:
                run_dir(0, "main", dx)
            dbuf = dx
        return (dbuf if ctx.needs_input_grad[0] else None, dh0, None, None, None, *wgrads)


class ReluRNN2Fn(Function):
    """bf16 tensor-core path of a multi-layer (bi)directional ReLU RNN with h_init = 0, one C call per layer
    (tacorl_rnn_layer2_{fwd,bwd}): both directions of a layer in one persistent launch, bf16 twins of every layer
    output / pre-activation gradient kept in the layer's own layout (no staging casts, no per-direction streams).
    grad_rows: only the first `grad_rows` batch rows ever receive a gradient (the action decoder batches a
    logging-only second plan behind the trained one): BPTT then runs on those rows alone."""

    @staticmethod
    def forward(ctx, x, num_layers, bidir, last_only, grad_rows, *weights):
        T, B, I = x.shape
        D = 2 if bidir else 1
        H = weights[1].shape[0]
        x = _c(x)
        weights = [_c(w) for w in weights]
        dev = x.device
        train = any(ctx.needs_input_grad)            # (grad mode itself is off inside forward)
        whts, prep_done = [None] * (num_layers * D), None
        if train:   # W_hh^T (the BPTT operand) on a side stream, under the latency-bound recurrence
            main, prep = torch.cuda.current_stream(dev), _prep_stream(dev)
            whts = [torch.empty(H, H, device=dev, dtype=torch.bfloat16) for _ in range(num_layers * D)]
            prep.wait_stream(main)
            with torch.cuda.stream(prep):
                for k in range(num_layers * D):
                    L.call("tacorl_cast_transpose_bf16", L.ptr(weights[k * 4 + 1]), H, H, L.ptr_any(whts[k]), L.stream())
                prep_done = torch.cuda.Event()
                prep_done.record(prep)
        outs, outbs = [], []
        inp, inp_b = x, None
        for l in range(num_layers):
            Il = inp.shape[2]
            out = torch.empty(T, B, D * H, device=dev, dtype=torch.float32)
            outb = torch.empty(T, B, D * H, device=dev, dtype=torch.bfloat16)
            wl = weights[l * D * 4:(l + 1) * D * 4]
            tw = []
            for d in range(D):
                tw += [shadow_of(wl[4 * d]), shadow_of(wl[4 * d + 1])]
            nst = [T] + ([1 if (last_only and l == num_layers - 1) else T] if D == 2 else [])
            ws = L.workspace(L.query("tacorl_rnn_layer2_ws_bytes", T, B, Il, H, D), dev, "main")
            L.call("tacorl_rnn_layer2_fwd", T, B, Il, H, D, L.ptr(inp), Il, L.ptr_any(inp_b), Il, L.ptr_array(wl),
                   L.ptr_array(tw), L.int_array(nst), L.ptr(out), D * H, L.ptr_any(outb),
                   ctypes.c_void_p(ws.data_ptr()), ws.numel(), L.stream())
            outs.append(out)
            outbs.append(outb)
            inp, inp_b = out, outb
        ctx.cfg = (T, B, I, H, D, num_layers, last_only, B if grad_rows is None else int(grad_rows))
        ctx.aux = (outbs, whts, prep_done)
        ctx.save_for_backward(x, *outs, *weights)
        if last_only:
            return inp[T - 1], None
        hn = torch.stack([outs[l][0 if d == 1 else T - 1, :, d * H:(d + 1) * H] for l in range(num_layers) for d in range(D)], 0)
        ctx.mark_non_differentiable(hn)
        return inp, hn

    @staticmethod
    def backward(ctx, d_out, _d_hn):
        T, B, I, H, D, num_layers, last_only, Bg = ctx.cfg
        saved = ctx.saved_tensors
        x = saved[0]
        outs = saved[1:1 + num_layers]
        weights = saved[1 + num_layers:]
        outbs, whts, prep_done = ctx.aux
        dev = x.device
        if last_only:
            dbuf = torch.zeros(T, B, D * H, device=dev, dtype=torch.float32)
            dbuf[T - 1].copy_(d_out)
        else:
            dbuf = d_out.contiguous().clone()
        if prep_done is not None:
            torch.cuda.current_stream(dev).wait_event(prep_done)
        wgrads = [None] * len(weights)
        for l in range(num_layers - 1, -1, -1):
            inp, inp_b = (x, None) if l == 0 else (outs[l - 1], outbs[l - 1])
            Il = inp.shape[2]
            need_dx = l > 0 or ctx.needs_input_grad[0]
            dx = torch.empty(T, B, Il, device=dev, dtype=torch.float32) if need_dx else None
            mk = torch.zeros if Bg < B else torch.empty       # rows without a gradient must read as zeros
            dpb = mk(T, B, D * H, device=dev, dtype=torch.bfloat16)
            wl = weights[l * D * 4:(l + 1) * D * 4]
            w2, tw, g = [], [], []
            for d in range(D):
                w2 += [wl[4 * d], wl[4 * d + 1]]
                tw += [shadow_of(wl[4 * d]), whts[l * D + d]]
                for j in range(4):   # straight into the optimiser's flat gradient when this is the parameter's first use
                    slot = grad_slot_of(wl[4 * d + j])
                    g.append(slot if slot is not None else torch.empty_like(wl[4 * d + j]))
            nst = [T] + ([1 if (last_only and l == num_layers - 1) else T] if D == 2 else [])
            ws = L.workspace(L.query("tacorl_rnn_layer2_ws_bytes", T, B, Il, H, D), dev, "main")
            L.call("tacorl_rnn_layer2_bwd", T, B, Bg, Il, H, D, L.ptr(inp), Il, L.ptr_any(inp_b), Il, L.ptr_array(w2),
                   L.ptr_array(tw), L.int_array(nst), L.ptr(outs[l]), D * H, L.ptr_any(outbs[l]), L.ptr(dbuf), D * H,
                   L.ptr_any(dpb), L.ptr(dx), Il, L.ptr_array(g), ctypes.c_void_p(ws.data_ptr()), ws.numel(), L.stream())
            wgrads[l * D * 4:(l + 1) * D * 4] = g
            dbuf = dx
        return (dbuf if ctx.needs_input_grad[0] else None, None, None, None, None, *wgrads)


def relu_rnn(x_tm, weights, num_layers, bidirectional, last_only=False, h0=None, grad_rows=None):
    if not torch.is_grad_enabled():
        # no backward will follow (validation, frozen encoders): keep no BPTT operands and fork no W_hh^T preparation
        # onto the prep stream, whose work only a backward joins (a captured graph would end with it unjoined)
        x_tm, weights = x_tm.detach(), [w.detach() for w in weights]
    if h0 is None and _STATE["prec"] == L.PREC_BF16 and x_tm.is_cuda and weights[1].shape[0] % 8 == 0:
        return ReluRNN2Fn.apply(x_tm, num_layers, bidirectional, last_only, grad_rows, *weights)
    return ReluRNNFn.apply(x_tm, h0, num_layers, bidirectional, last_only, *weights)


# --------------------------------------------------------------------------------------- losses
class DlmLossFn(Function):
    """Discretised logistic mixture NLL + gripper CE (mean over rows)."""

    @staticmethod
    def forward(ctx, logits, actions, num_classes, act_min, act_max, gripper_alpha):
        logits, actions = _c(logits), _c(actions)
        rows, A = logits.shape[0], actions.shape[1] - 1
        assert logits.shape[1] == 3 * A * 10 + 2
        dev = logits.device
        row_loss = torch.empty(rows * (A + 1), device=dev)
        loss = torch.empty(1, device=dev)
        need = ctx.needs_input_grad[0]
        dlog = torch.empty_like(logits) if need else None
        L.call("tacorl_dlm_nll", rows, A, L.ptr(logits), logits.shape[1], L.ptr(actions), actions.shape[1],
               int(num_classes), float(act_min), float(act_max), float(gripper_alpha), L.ptr(row_loss), L.ptr(loss),
               L.ptr(dlog), logits.shape[1], L.stream())
        if need:
            ctx.save_for_backward(dlog)
        return loss.view(())

    @staticmethod
    def backward(ctx, g):
        (dlog,) = ctx.saved_tensors
        return scale(dlog, _c(g.reshape(1))), None, None, None, None, None


def dlm_loss(logits, actions, num_classes=10, act_min=-1.0, act_max=1.0, gripper_alpha=1.0):
    return DlmLossFn.apply(logits, actions, num_classes, act_min, act_max, gripper_alpha)


def dlm_sample(logits, u1, u2, actions=None, grip_lo=-1.0, grip_hi=1.0):
    """Returns (pred (rows, A+1), gripper accuracy scalar or None).  No gradient."""
    logits = _c(logits.detach())
    rows = logits.shape[0]
    A = (logits.shape[1] - 2) // 30
    dev = logits.device
    pred = torch.empty(rows, A + 1, device=dev)
    hit = torch.empty(rows, device=dev) if actions is not None else None
    acc = torch.empty(1, device=dev) if actions is not None else None
    actions_c = _c(actions) if actions is not None else None
    u1, u2 = _c(u1), _c(u2)          # keep the (possibly copied) operands alive until the launch is enqueued
    L.call("tacorl_dlm_sample", rows, A, L.ptr(logits), logits.shape[1], L.ptr(u1), L.ptr(u2),
           L.ptr(actions_c), actions_c.shape[1] if actions is not None else 0, float(grip_lo), float(grip_hi),
           L.ptr(pred), L.ptr(hit), L.ptr(acc), L.stream())
    return pred, (acc.view(()) if acc is not None else None)


class GaussHeadFn(Function):
    """raw (rows, 2L) -> mean = clamp(+-9), std = exp(clamp(-5, 2))  (MLPPolicy.forward)."""

    @staticmethod
    def forward(ctx, raw):
        raw = _c(raw)
        rows, L2 = raw.shape
        mean = torch.empty(rows, L2 // 2, device=raw.device)
        std = torch.empty_like(mean)
        L.call("tacorl_gauss_head_fwd", rows, L2 // 2, L.ptr(raw), L.ptr(mean), L.ptr(std), L.stream())
        ctx.save_for_backward(raw, std)
        return mean, std

    @staticmethod
    def backward(ctx, dmean, dstd):
        raw, std = ctx.saved_tensors
        draw = torch.empty_like(raw)
        dmean = _c(dmean) if dmean is not None else None
        dstd = _c(dstd) if dstd is not None else None
        L.call("tacorl_gauss_head_bwd", raw.shape[0], raw.shape[1] // 2, L.ptr(raw), L.ptr(std),
               L.ptr(dmean), L.ptr(dstd), L.ptr(draw), L.stream())
        return draw


class SoftplusHeadFn(Function):
    """raw (rows, 2L) -> mean, std = softplus(var) + min_std  (plan recognition heads)."""

    @staticmethod
    def forward(ctx, raw, min_std):
        raw = _c(raw)
        rows, L2 = raw.shape
        mean = torch.empty(rows, L2 // 2, device=raw.device)
        std = torch.empty_like(mean)
        L.call("tacorl_softplus_head_fwd", rows, L2 // 2, L.ptr(raw), float(min_std), L.ptr(mean), L.ptr(std),
               L.stream())
        ctx.save_for_backward(raw)
        return mean, std

    @staticmethod
    def backward(ctx, dmean, dstd):
        (raw,) = ctx.saved_tensors
        draw = torch.empty_like(raw)
        dmean = _c(dmean) if dmean is not None else None
        dstd = _c(dstd) if dstd is not None else None
        L.call("tacorl_softplus_head_bwd", raw.shape[0], raw.shape[1] // 2, L.ptr(raw), L.ptr(dmean), L.ptr(dstd),
               L.ptr(draw), L.stream())
        return draw, None


def gauss_head(raw):
    return GaussHeadFn.apply(raw)


def softplus_head(raw, min_std):
    return SoftplusHeadFn.apply(raw, min_std)


class KLBalancedFn(Function):
    @staticmethod
    def forward(ctx, mu_q, sd_q, mu_p, sd_p, kl_alpha, balancing):
        mu_q, sd_q, mu_p, sd_p = _c(mu_q), _c(sd_q), _c(mu_p), _c(sd_p)
        B, Ld = mu_q.shape
        kl = torch.empty(1, device=mu_q.device)
        gs = [torch.empty_like(mu_q) for _ in range(4)]
        L.call("tacorl_kl_balanced", B, Ld, L.ptr(mu_q), L.ptr(sd_q), L.ptr(mu_p), L.ptr(sd_p), float(kl_alpha),
               int(balancing), L.ptr(kl), L.ptr(gs[0]), L.ptr(gs[1]), L.ptr(gs[2]), L.ptr(gs[3]), L.stream())
        ctx.save_for_backward(*gs)
        return kl.view(())

    @staticmethod
    def backward(ctx, g):
        g = _c(g.reshape(1))
        return (*[scale(t, g) for t in ctx.saved_tensors], None, None)


def kl_balanced(mu_q, sd_q, mu_p, sd_p, kl_alpha=0.8, balancing=True):
    return KLBalancedFn.apply(mu_q, sd_q, mu_p, sd_p, kl_alpha, balancing)


class TanhRsampleFn(Function):
    """a = tanh(mu + std*eps) (or the raw z when apply_tanh=False); also returns z."""

    @staticmethod
    def forward(ctx, mu, sd, eps, apply_tanh):
        mu, sd, eps = _c(mu), _c(sd), _c(eps)
        a = torch.empty_like(eps)
        z = torch.empty_like(eps)
        L.call("tacorl_tanh_rsample_fwd", eps.numel(), mu.numel(), L.ptr(mu), L.ptr(sd), L.ptr(eps), L.ptr(a),
               L.ptr(z), int(apply_tanh), L.stream())
        ctx.apply_tanh = apply_tanh
        ctx.same = eps.numel() == mu.numel()
        ctx.save_for_backward(a, eps)
        return a, z

    @staticmethod
    def backward(ctx, da, dz):
        a, eps = ctx.saved_tensors
        assert ctx.same, "gradient through sample_n broadcasting is not used by the reference"
        dmu = torch.empty_like(a)
        dsd = torch.empty_like(a)
        da = _c(da) if da is not None else None
        dz = _c(dz) if dz is not None else None
        L.call("tacorl_tanh_rsample_bwd", a.numel(), L.ptr(a), L.ptr(eps), L.ptr(da), L.ptr(dz), L.ptr(dmu), L.ptr(dsd),
               int(ctx.apply_tanh), L.stream())
        return dmu, dsd, None, None


def tanh_rsample(mu, sd, eps, apply_tanh=True):
    return TanhRsampleFn.apply(mu, sd, eps, apply_tanh)


class TanhLogProbFn(Function):
    """TanhNormal.log_prob -> (rows, 1).  z is the pre-tanh value, or the tanh'ed value when from_value."""

    @staticmethod
    def forward(ctx, mu, sd, z, from_value):
        mu, sd, z = _c(mu), _c(sd), _c(z)
        Ld = z.shape[-1]
        rows = z.numel() // Ld
        brows = mu.numel() // Ld
        logp = torch.empty(rows, device=z.device)
        need = any(ctx.needs_input_grad[:3])
        g = [torch.empty_like(z) for _ in range(3)] if need else [None] * 3
        L.call("tacorl_tanh_logprob", rows, Ld, brows, L.ptr(mu), L.ptr(sd), L.ptr(z), int(from_value), L.ptr(logp),
               L.ptr(g[0]), L.ptr(g[1]), L.ptr(g[2]), L.stream())
        if need:
            assert rows == brows, "gradient through a broadcast log_prob is not used by the reference"
            ctx.save_for_backward(*g)
        ctx.from_value = from_value
        ctx.Ld = Ld
        return logp.view(*z.shape[:-1], 1)

    @staticmethod
    def backward(ctx, dlogp):
        gmu, gsd, gz = ctx.saved_tensors
        d = _c(dlogp.reshape(-1))
        rows = d.numel()

        def rs(t):
            o = torch.empty_like(t)
            L.call("tacorl_rowscale", rows, ctx.Ld, L.ptr(t), L.ptr(d), 1.0, L.ptr(o), 0, L.stream())
            return o

        return (rs(gmu) if ctx.needs_input_grad[0] else None, rs(gsd) if ctx.needs_input_grad[1] else None,
                rs(gz) if (ctx.needs_input_grad[2] and not ctx.from_value) else None, None)


def tanh_logprob(mu, sd, z, from_value=False):
    return TanhLogProbFn.apply(mu, sd, z, from_value)


# --------------------------------------------------------------------------------------- discrete gripper head
def gripper_gumbel(logits, u, clamp):
    """Class index (0 / 1, float, shape u.shape[:-1] + (1,)) drawn by GumbelSoftmax(logits) from the uniforms u
    (tacorl_gripper_gumbel; no gradient: the reference keeps only the argmax of a draw, actor.py:84-91)."""
    logits, u = _c(logits.detach()), _c(u)
    rows, rows0 = u.numel() // 2, logits.numel() // 2
    index = torch.empty(rows, device=u.device, dtype=torch.float32)
    L.call("tacorl_gripper_gumbel", rows, rows0, L.ptr(logits), L.ptr(u), int(clamp), L.ptr(index), None, L.stream())
    return index.view(*u.shape[:-1], 1)


class GripperLogProbFn(Function):
    """GumbelSoftmax.log_prob of class indices (distributions.py:50-58) -> (..., 1); gradient w.r.t. the logits."""

    @staticmethod
    def forward(ctx, logits, index):
        logits, index = _c(logits), _c(index.to(torch.float32))
        rows, rows0 = index.numel(), logits.numel() // 2
        logp = torch.empty(rows, device=logits.device, dtype=torch.float32)
        L.call("tacorl_gripper_logprob", rows, rows0, L.ptr(logits), L.ptr(index), L.ptr(logp), L.stream())
        if ctx.needs_input_grad[0]:
            assert rows == rows0, "gradient through a broadcast gripper log_prob is not used by the reference"
            ctx.save_for_backward(logits, index)
        lead = index.shape[:-1] if index.dim() > 1 and index.shape[-1] == 1 else index.shape
        return logp.view(*lead, 1)

    @staticmethod
    def backward(ctx, dlogp):
        logits, index = ctx.saved_tensors
        d = _c(dlogp.reshape(-1))
        dlogits = torch.empty_like(logits)
        L.call("tacorl_gripper_logprob_bwd", d.numel(), L.ptr(logits), L.ptr(index), L.ptr(d), L.ptr(dlogits), L.stream())
        return dlogits, None


def gripper_logprob(logits, index):
    return GripperLogProbFn.apply(logits, index)


# --------------------------------------------------------------------------------------- CQL
CQL_SCALARS = ("bellman_q1_loss", "bellman_q2_loss", "conservative_q1_loss", "conservative_q2_loss",
               "alpha_prime", "alpha_prime_loss", "q1_loss", "q2_loss", "q1_data", "q1_random", "q1_policy",
               "q2_data", "q2_random", "q2_policy")


class CqlCriticLossFn(Function):
    """Returns (q1_loss, q2_loss, scalars[14], d_log_alpha_prime).  Gradients flow to q1_all / q2_all only
    (log_alpha_prime's own gradient — of alpha_prime_loss — is returned as a value, because the reference
    steps alpha' from that loss alone and discards what the q-losses deposit, SURVEY Appendix E.6)."""

    @staticmethod
    def forward(ctx, q1_all, q2_all, lp_curr, lp_next, tq1, tq2, reward, done, log_alpha_prime, n, rand_density,
                discount, reward_scale, gap, cw, temp, with_lagrange):
        ctx.qshapes = (q1_all.shape, q2_all.shape)
        q1_all, q2_all = _c(q1_all.reshape(-1)), _c(q2_all.reshape(-1))
        B = tq1.numel()
        dev = q1_all.device
        scal = torch.empty(14, device=dev)
        dq1, dq2 = torch.empty_like(q1_all), torch.empty_like(q2_all)
        dlap = torch.empty(1, device=dev)
        lp_curr, lp_next = _c(lp_curr.reshape(-1)), _c(lp_next.reshape(-1))
        tq1, tq2 = _c(tq1.reshape(-1)), _c(tq2.reshape(-1))
        reward, done = _c(reward.reshape(-1)), _c(done.reshape(-1))
        L.call("tacorl_cql_critic_loss", B, n, L.ptr(q1_all), L.ptr(q2_all), L.ptr(lp_curr),
               L.ptr(lp_next), L.ptr(tq1), L.ptr(tq2),
               L.ptr(reward), L.ptr(done),
               L.ptr(log_alpha_prime) if with_lagrange else None, float(rand_density), float(discount),
               float(reward_scale), float(gap), float(cw), float(temp), int(with_lagrange), L.ptr(scal),
               L.ptr(dq1), L.ptr(dq2), L.ptr(dlap), L.stream())
        ctx.save_for_backward(dq1, dq2)
        ctx.mark_non_differentiable(scal, dlap)
        return scal[6].clone(), scal[7].clone(), scal, dlap

    @staticmethod
    def backward(ctx, g1, g2, _gs, _gl):
        dq1, dq2 = ctx.saved_tensors
        r1 = scale(dq1, _c(g1.reshape(1))).view(ctx.qshapes[0]) if g1 is not None else None
        r2 = scale(dq2, _c(g2.reshape(1))).view(ctx.qshapes[1]) if g2 is not None else None
        return (r1, r2) + (None,) * 15


class CqlActorLossFn(Function):
    """mode 1: mean(alpha*log_pi - a); mode 2: mean(alpha*log_pi - min(a, b)).  alpha = exp(log_alpha) is
    treated as a constant (its deposit is discarded by the reference, Appendix E.6)."""

    @staticmethod
    def forward(ctx, mode, log_pi, a, b, log_alpha):
        ctx.in_shapes = (log_pi.shape, a.shape, b.shape if b is not None else None)
        log_pi, a = _c(log_pi.reshape(-1)), _c(a.reshape(-1))
        b = _c(b.reshape(-1)) if b is not None else None
        B = log_pi.numel()
        dev = log_pi.device
        out = torch.empty(2, device=dev)
        dlp, da = torch.empty_like(log_pi), torch.empty_like(a)
        db = torch.empty_like(b) if b is not None else None
        L.call("tacorl_cql_actor_loss", mode, B, L.ptr(log_pi), L.ptr(a), L.ptr(b), L.ptr(log_alpha), 0.0,
               L.ptr(out), None, L.ptr(dlp), L.ptr(da), L.ptr(db), L.stream())
        ctx.save_for_backward(dlp, da, db)
        ctx.shapes = None
        ctx.mark_non_differentiable(out)
        return out[0].clone(), out

    @staticmethod
    def backward(ctx, g, _go):
        dlp, da, db = ctx.saved_tensors
        g = _c(g.reshape(1))
        sh = ctx.in_shapes
        return (None, scale(dlp, g).view(sh[0]), scale(da, g).view(sh[1]),
                scale(db, g).view(sh[2]) if db is not None else None, None)


def cql_alpha_loss(log_pi, log_alpha, target_entropy):
    """Returns (alpha_loss value (1,), d alpha_loss / d log_alpha (1,)) — plain values, no graph."""
    log_pi = _c(log_pi.detach().reshape(-1))
    out = torch.empty(2, device=log_pi.device)
    dla = torch.empty(1, device=log_pi.device)
    L.call("tacorl_cql_actor_loss", 0, log_pi.numel(), L.ptr(log_pi), None, None, L.ptr(log_alpha),
           float(target_entropy), L.ptr(out), L.ptr(dla), None, None, None, L.stream())
    return out[:1], dla


# --------------------------------------------------------------------------------------- optimiser kernels
def adam_step(p, g, m, v, lr, step, beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=1.0, sqnorm=None, max_norm=0.0,
              step_dev=None, shadow=None, increment=True, background=False):
    """step_dev: optional int32 device tensor holding the step count (incremented by the call unless increment=False:
    the later slices of a step that is applied slice by slice).
    shadow: optional bf16 tensor of p.numel() elements that receives a bf16 copy of the updated parameters.
    background: small grid that shares the SMs with concurrently running kernels (the early slice of FlatAdam)."""
    sd = ctypes.c_void_p(step_dev.data_ptr()) if step_dev is not None else None
    L.call("tacorl_adam_step_range", p.numel(), L.ptr(p), L.ptr(g), L.ptr(m), L.ptr(v), float(lr), float(beta1),
           float(beta2), float(eps), int(step), sd, int(increment), int(background), float(grad_scale), L.ptr(sqnorm),
           float(max_norm), L.ptr_any(shadow), L.stream())


def polyak_update(target, source, tau):
    L.call("tacorl_polyak_update", target.numel(), L.ptr(target), L.ptr(source), float(tau), L.stream())


def sqnorm(x, out=None):
    if out is None:
        out = torch.empty(1, device=x.device)
    ws = torch.empty(592, device=x.device)
    L.call("tacorl_sqnorm", x.numel(), L.ptr(x), L.ptr(out), L.ptr(ws), L.stream())
    return out


# --------------------------------------------------------------------------------------- transformer pieces
class PosEmbFn(Function):
    """x (T,B,D) = (emb (B,T,D0) zero-padded to D + pos[:T]) * mask."""

    @staticmethod
    def forward(ctx, emb, pos, mask):
        emb, pos = _c(emb), _c(pos)
        B, T, D0 = emb.shape
        D = pos.shape[1]
        x = torch.empty(T, B, D, device=emb.device)
        L.call("tacorl_posemb_fwd", B, T, D0, D, L.ptr(emb), L.ptr(pos), L.ptr(mask), L.ptr(x), L.stream())
        ctx.dims = (B, T, D0, D, pos.shape[0])
        ctx.save_for_backward(mask)
        return x

    @staticmethod
    def backward(ctx, dx):
        (mask,) = ctx.saved_tensors
        B, T, D0, D, npos = ctx.dims
        demb = torch.empty(B, T, D0, device=dx.device) if ctx.needs_input_grad[0] else None
        dpos = torch.zeros(npos, D, device=dx.device)
        L.call("tacorl_posemb_bwd", B, T, D0, D, L.ptr(_c(dx)), L.ptr(mask), L.ptr(demb), L.ptr(dpos), L.stream())
        return demb, dpos, None


class AttentionFn(Function):
    """Multi-head self-attention core on packed qkv (T,B,3D) -> (T,B,D)."""

    @staticmethod
    def forward(ctx, qkv, heads, amask):
        qkv = _c(qkv)
        T, B, D3 = qkv.shape
        D = D3 // 3
        P = torch.empty(B * heads, T, T, device=qkv.device)
        out = torch.empty(T, B, D, device=qkv.device)
        L.call("tacorl_attn_fwd", B, T, D, heads, L.ptr(qkv), L.ptr(amask), L.ptr(P), L.ptr(out), L.stream())
        ctx.heads = heads
        ctx.save_for_backward(qkv, amask, P)
        return out

    @staticmethod
    def backward(ctx, dout):
        qkv, amask, P = ctx.saved_tensors
        T, B, D3 = qkv.shape
        dqkv = torch.empty_like(qkv)
        L.call("tacorl_attn_bwd", B, T, D3 // 3, ctx.heads, L.ptr(qkv), L.ptr(amask), L.ptr(P), L.ptr(_c(dout)),
               L.ptr(dqkv), L.stream())
        return dqkv, None, None


class AddLayerNormFn(Function):
    """LayerNorm(x + r*mask) over the last dim (post-norm residual block)."""

    @staticmethod
    def forward(ctx, x, r, mask, w, b, eps):
        x, r = _c(x), _c(r)
        D = x.shape[-1]
        rows = x.numel() // D
        y, xhat = torch.empty_like(x), torch.empty_like(x)
        rstd = torch.empty(rows, device=x.device)
        w, b = _c(w), _c(b)
        L.call("tacorl_add_ln_fwd", rows, D, L.ptr(x), L.ptr(r), L.ptr(mask), L.ptr(w), L.ptr(b), float(eps),
               L.ptr(y), L.ptr(xhat), L.ptr(rstd), L.stream())
        ctx.save_for_backward(xhat, rstd, w, mask)
        return y

    @staticmethod
    def backward(ctx, dy):
        xhat, rstd, w, mask = ctx.saved_tensors
        D = xhat.shape[-1]
        rows = xhat.numel() // D
        dx, dr = torch.empty_like(xhat), torch.empty_like(xhat)
        dw, db = torch.zeros(D, device=dy.device), torch.zeros(D, device=dy.device)
        dy, w = _c(dy), _c(w)
        L.call("tacorl_add_ln_bwd", rows, D, L.ptr(dy), L.ptr(xhat), L.ptr(rstd), L.ptr(w), L.ptr(mask),
               L.ptr(dx), L.ptr(dr), L.ptr(dw), L.ptr(db), L.stream())
        return dx, dr, None, dw, db, None


class MeanTimeFn(Function):
    @staticmethod
    def forward(ctx, x):
        x = _c(x)
        B, T, C = x.shape
        y = torch.empty(B, C, device=x.device)
        L.call("tacorl_mean_t_fwd", B, T, C, L.ptr(x), L.ptr(y), L.stream())
        ctx.dims = (B, T, C)
        return y

    @staticmethod
    def backward(ctx, dy):
        B, T, C = ctx.dims
        dx = torch.empty(B, T, C, device=dy.device)
        L.call("tacorl_mean_t_bwd", B, T, C, L.ptr(_c(dy)), L.ptr(dx), L.stream())
        return dx


class MaskMulFn(Function):
    """x * mask (dropout with an explicit pre-scaled keep mask)."""

    @staticmethod
    def forward(ctx, x, mask):
        x = _c(x)
        out = torch.empty_like(x)
        L.call("tacorl_mul", x.numel(), L.ptr(x), L.ptr(mask), L.ptr(out), L.stream())
        ctx.save_for_backward(mask)
        return out

    @staticmethod
    def backward(ctx, dy):
        (mask,) = ctx.saved_tensors
        dy = _c(dy)
        dx = torch.empty_like(dy)
        L.call("tacorl_mul", dy.numel(), L.ptr(dy), L.ptr(mask), L.ptr(dx), L.stream())
        return dx, None


def posemb(emb, pos, mask=None):
    return PosEmbFn.apply(emb, pos, mask)


def attention(qkv, heads, amask=None):
    return AttentionFn.apply(qkv, heads, amask)


def add_layernorm(x, r, w, b, mask=None, eps=1e-5):
    return AddLayerNormFn.apply(x, r, mask, w, b, eps)


def mean_time(x):
    return MeanTimeFn.apply(x)


def mask_mul(x, mask):
    return x if mask is None else MaskMulFn.apply(x, mask)
