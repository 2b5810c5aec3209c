"""ReluRNN2Fn's backward with each layer's weight gradients on a second stream, beside the next layer's BPTT.

The weight-gradient kernels are the ones the one-call tacorl_rnn_layer2_bwd runs, with the same split-K counts; only the
stream and the persistent GEMM grid (TcArgs::max_ctas) differ, and the grid decides which CTA computes a tile, not how
a tile is summed.  So every gradient must equal, bit for bit, the same layers run one tacorl_rnn_layer2_bwd call at a time
with a device synchronise between calls.  Shapes are the flagship step's: the action decoder (2 layers, batch 128 of
which the first 64 rows carry a gradient) and the plan recogniser (2 bidirectional layers, last_only)."""
import ctypes

import pytest
import torch

from tacorl_b200 import ops

DEV = "cuda"
H = 2048
DECODER = dict(T=15, B=128, I=48, D=1, last_only=False, grad_rows=64)
RECOGNISER = dict(T=16, B=64, I=64, D=2, last_only=True, grad_rows=None)


def test_wgrad_cta_cap_leaves_the_recurrence_its_sms():
    assert ops.wgrad_cta_cap(0) == 148                  # nothing beside it: one CTA per SM
    assert ops.wgrad_cta_cap(1) == 84                   # one lane: 64 SMs taken
    assert ops.wgrad_cta_cap(2) == 20                   # two lanes: 128 SMs taken
    assert ops.wgrad_cta_cap(3) == 1                    # never an empty grid
    for lanes in (1, 2):
        assert ops.wgrad_cta_cap(lanes) + 64 * lanes <= 148


def _vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _same(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _weights(g, cfg):
    D = cfg["D"]
    w = []
    for l in range(2):
        I = cfg["I"] if l == 0 else D * H
        for _ in range(D):
            k = H ** -0.5
            w += [(torch.rand(H, I, generator=g) * 2 - 1) * k, (torch.rand(H, H, generator=g) * 2 - 1) * k,
                  (torch.rand(H, generator=g) * 2 - 1) * k, (torch.rand(H, generator=g) * 2 - 1) * k]
    return [t.to(DEV) for t in w]


def _cotangent(g, cfg):
    T, B, D = cfg["T"], cfg["B"], cfg["D"]
    cot = torch.randn(B, D * H, generator=g) if cfg["last_only"] else torch.randn(T, B, D * H, generator=g)
    if cfg["grad_rows"]:
        cot[..., cfg["grad_rows"]:, :] = 0
    return cot.to(DEV)


def _abi_chain(L, x, w, cfg, cot):
    """Input and weight gradients of the 2-layer network through one tacorl_rnn_layer2_bwd call per layer, each
    followed by a device synchronise."""
    T, B, D = cfg["T"], cfg["B"], cfg["D"]
    Bg = cfg["grad_rows"] or 0
    outs, inp, inp_b = [], x, None
    for l in range(2):
        Il = inp.shape[2]
        out = torch.empty(T, B, D * H, device=DEV)
        outb = torch.empty(T, B, D * H, device=DEV, dtype=torch.bfloat16)
        nst = [T] + ([1 if (cfg["last_only"] and l == 1) else T] if D == 2 else [])
        buf = torch.empty(L.query("tacorl_rnn_layer2_ws_bytes", T, B, Il, H, D), dtype=torch.uint8, device=DEV)
        L.call("tacorl_rnn_layer2_fwd", T, B, Il, H, D, _vp(inp), Il, _vp(inp_b), Il, L.ptr_array(w[4 * D * l:4 * D * (l + 1)]),
               None, L.int_array(nst), _vp(out), D * H, _vp(outb), _vp(buf), buf.numel(), L.stream())
        outs.append((inp, inp_b, out, outb, nst))
        inp, inp_b = out, outb
    if cfg["last_only"]:
        dbuf = torch.zeros(T, B, D * H, device=DEV)
        dbuf[T - 1] = cot
    else:
        dbuf = cot.clone()
    grads = [None] * len(w)
    for l in (1, 0):
        inp, inp_b, out, outb, nst = outs[l]
        Il = inp.shape[2]
        wl = w[4 * D * l:4 * D * (l + 1)]
        w2 = [wl[4 * d + j] for d in range(D) for j in (0, 1)]
        dpb = torch.zeros(T, B, D * H, device=DEV, dtype=torch.bfloat16)
        dx = torch.empty(T, B, Il, device=DEV)
        dw = [torch.empty_like(t) for t in wl]
        buf = torch.empty(L.query("tacorl_rnn_layer2_ws_bytes", T, B, Il, H, D), dtype=torch.uint8, device=DEV)
        L.call("tacorl_rnn_layer2_bwd", T, B, Bg, Il, H, D, _vp(inp), Il, _vp(inp_b), Il, L.ptr_array(w2), None,
               L.int_array(nst), _vp(out), D * H, _vp(outb), _vp(dbuf), D * H, _vp(dpb), _vp(dx), Il, L.ptr_array(dw),
               _vp(buf), buf.numel(), L.stream())
        torch.cuda.synchronize()
        grads[4 * D * l:4 * D * (l + 1)] = dw
        dbuf = dx
    return dbuf, grads


@pytest.fixture
def bf16():
    from tacorl_b200 import _lib
    lib = _lib.lib()
    was_prec = ops.get_precision()
    was_seq = lib.tacorl_rnn_seq_enable(1)
    ops.set_precision("bf16")
    t0 = lib.tacorl_rnn_seq_timeouts()
    yield _lib
    assert lib.tacorl_rnn_seq_timeouts() == t0          # no recurrence ever waited on a co-resident peer in vain
    lib.tacorl_rnn_seq_enable(was_seq)
    ops.set_precision(was_prec)


def _run(x, params, cfg, cot):
    y, _ = ops.relu_rnn(x, list(params), 2, cfg["D"] == 2, cfg["last_only"], grad_rows=cfg["grad_rows"])
    (y * cot).sum().backward()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["decoder", "recogniser"])
def test_overlapped_backward_is_the_one_call_chain(bf16, name):
    from tacorl_b200.optim import FlatAdam
    L = bf16
    cfg = DECODER if name == "decoder" else RECOGNISER
    g = torch.Generator().manual_seed(5)
    w = _weights(g, cfg)
    x = torch.randn(cfg["T"], cfg["B"], cfg["I"], generator=g).to(DEV)
    cot = _cotangent(g, cfg)
    dx_ref, ref = _abi_chain(L, x, w, cfg, cot)
    params = [torch.nn.Parameter(t.clone()) for t in w]
    opt = FlatAdam(params, lr=1e-4)
    xd = x.clone().requires_grad_(True)
    torch.cuda.synchronize()
    _run(xd, params, cfg, cot)
    # read on the current stream with no synchronise in between: the backward pass has joined the weight gradients
    got = [p.grad.clone() for p in params]
    got_dx = xd.grad.clone()
    torch.cuda.synchronize()
    for i, (p, gv) in enumerate(zip(params, opt.grad_views)):
        assert p.grad.data_ptr() == gv.data_ptr(), i       # written straight into the flat gradient (the deferred path)
    assert not ops._PENDING                                # ... and joined when the backward pass ended
    assert _same(got_dx, dx_ref)
    for i, (a, b) in enumerate(zip(got, ref)):
        assert _same(a, b), i


@pytest.mark.gpu
def test_second_backward_without_zero_grad_accumulates(bf16):
    """The second pass finds the slots taken: its gradients are temporaries, joined before the backward returns, and
    autograd adds them to .grad."""
    from tacorl_b200.optim import FlatAdam
    L = bf16
    cfg = DECODER
    g = torch.Generator().manual_seed(6)
    w = _weights(g, cfg)
    x = torch.randn(cfg["T"], cfg["B"], cfg["I"], generator=g).to(DEV)
    cots = [_cotangent(g, cfg), _cotangent(g, cfg)]
    refs = [_abi_chain(L, x, w, cfg, c)[1] for c in cots]
    params = [torch.nn.Parameter(t.clone()) for t in w]
    FlatAdam(params, lr=1e-4)
    for c in cots:
        _run(x, params, cfg, c)
    got = [p.grad.clone() for p in params]
    torch.cuda.synchronize()
    for i, (a, r0, r1) in enumerate(zip(got, *refs)):
        assert _same(a, r0 + r1), i


@pytest.mark.gpu
def test_captured_step_replays_the_eager_step(bf16):
    """zero_grad, forward, backward and FlatAdam.step captured in a CUDA graph (the capture ends with the wgrad stream
    joined) give, on replay, the parameters and moments of the same step run eagerly."""
    from tacorl_b200.optim import FlatAdam
    cfg = RECOGNISER
    g = torch.Generator().manual_seed(8)
    w = _weights(g, cfg)
    x = torch.randn(cfg["T"], cfg["B"], cfg["I"], generator=g).to(DEV)
    cot = _cotangent(g, cfg)
    params = [torch.nn.Parameter(t.clone()) for t in w]
    opt = FlatAdam(params, lr=1e-3)

    def step():
        opt.zero_grad(set_to_none=True)
        _run(x, params, cfg, cot)
        opt.step()

    snap = opt.snapshot()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()                                         # warm-up: workspaces and streams exist before the capture
    torch.cuda.current_stream().wait_stream(side)
    eager = (opt.flat_params.clone(), opt.exp_avg.clone(), opt.exp_avg_sq.clone())
    opt.restore(snap)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    opt.restore(snap)
    torch.cuda.synchronize()
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, (opt.flat_params, opt.exp_avg, opt.exp_avg_sq)):
        assert _same(a, b)


@pytest.mark.gpu
def test_graphed_bf16_play_lmp_step_replays_the_eager_step(bf16):
    """The flagship step: bf16 PlayLMP through runtime.play_lmp_step_fn (early Adam on: the embeddings' hook updates the
    slice behind the encoders on its own stream, which must wait for the recogniser's weight gradients still running on
    the wgrad stream; goal encoder and plan proposal on the forked plan stream), captured by GraphedTrainStep.  One
    replay leaves the parameters, moments and bf16 twins of one eager step, bit for bit."""
    from oracle import synth as S
    from tacorl_b200 import runtime
    from tests.gpu_util import build_play_lmp, to_dev
    B, T, HW = 64, 16, 84
    m = build_play_lmp("tanh_net", ("rgb_static",), H, 16, T)
    shapes = {k: list(v.shape) for k, v in m.state_dict().items()}
    m.load_state_dict(S.synth_state_dict(shapes, 4))
    m.to(DEV)
    opt = m.configure_optimizers()
    batch = to_dev(S.synth_play_batch(B, T, HW, HW, 4))
    batch = {"states": batch["states"], "actions": batch["actions"]}
    fn = runtime.play_lmp_step_fn(m, opt)
    assert opt.early_step
    snap = opt.snapshot()
    torch.manual_seed(11)
    fn(batch)
    torch.cuda.synchronize()
    eager = (opt.flat_params.clone(), opt.exp_avg.clone(), opt.exp_avg_sq.clone(), opt.shadow.clone())
    assert not ops._PENDING
    opt.restore(snap)
    g = runtime.GraphedTrainStep(fn, batch, warmup=2)        # (its warm-up steps are rolled back)
    torch.manual_seed(11)                                     # the replay draws the eager step's noise
    g()
    torch.cuda.synchronize()
    assert int(opt._step_dev) == 1
    for a, b in zip(eager, (opt.flat_params, opt.exp_avg, opt.exp_avg_sq, opt.shadow)):
        assert torch.equal(a.view(torch.int16 if a.element_size() == 2 else torch.int32),
                           b.view(torch.int16 if b.element_size() == 2 else torch.int32))
