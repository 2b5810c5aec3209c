"""The GEMM oracle (tests/gemm_oracle.py) checked on the CPU before any GPU is involved:
  - its fp64 formulas reproduce torch's fp64 addmm / relu / silu / masking for every operand layout and epilogue;
  - a torch emulation of the kernels' arithmetic (bf16-exact operands, fp32 accumulation, split-K partials summed in
    fp32, fp32 epilogue, bf16 rounding of Cb) passes the check at the tolerance the GPU tests use;
  - every discrimination control, and a one-ulp change of one element of Cb, fails it by at least 20x that tolerance;
  - the Python copy of the dispatch rules predicts the route of every case of the GPU table."""
import pytest
import torch
import torch.nn.functional as F

from tests import gemm_oracle as G
from tests.gemm_oracle import TAU


def emulate(A, B, a_mn, b_mn, splits=1, alpha=1.0, beta=0.0, C0=None, bias=None, act=G.ACT_NONE, gate=None):
    """The kernels' arithmetic in fp32: per K slice an fp32 product of the exact operands, the slices summed in order,
    then alpha, beta * C0, bias, act, gate in fp32 and the bf16 copy.  Returns (pre, out, out_bf16)."""
    a, b = G.op_a(A, a_mn).float(), G.op_b(B, b_mn).float()
    K = a.shape[1]
    per = G.cdiv(G.cdiv(K, G.BK), splits) * G.BK
    acc = torch.zeros(a.shape[0], b.shape[1])
    for k0 in range(0, K, per):
        acc = acc + a[:, k0:k0 + per] @ b[k0:k0 + per]
    v = alpha * acc
    if beta != 0:
        v = v + beta * C0
    if bias is not None:
        v = v + bias
    pre = v
    v = torch.relu(v) if act == G.ACT_RELU else (F.silu(v) if act == G.ACT_SILU else v)
    if gate is not None:
        v = torch.where(gate <= 0, torch.zeros_like(v), v)
    return pre, v, v.bfloat16()


def _fields(ep, C0, bias, gate):
    return dict(alpha=ep.get("alpha", 1.0), beta=ep.get("beta", 0.0), C0=C0 if ep.get("beta") else None,
                bias=bias if ep.get("bias") else None, act=ep.get("act", G.ACT_NONE), gate=gate if ep.get("gate") else None)


@pytest.mark.parametrize("layout", list(G.LAYOUTS))
@pytest.mark.parametrize("epi", list(G.EPILOGUES))
def test_oracle_matches_torch_fp64(layout, epi):
    a_mn, b_mn = G.LAYOUTS[layout]
    g = torch.Generator().manual_seed(11)
    M, N, K = 37, 29, 75
    A = torch.randn((K, M) if a_mn else (M, K), generator=g, dtype=torch.float64)
    B = torch.randn((K, N) if b_mn else (N, K), generator=g, dtype=torch.float64)
    C0, bias, gate = G.make_epilogue_inputs(g, M, N, K)
    f = _fields(G.EPILOGUES[epi], C0.double(), bias.double(), gate.double())
    ref = G.reference(G.Products(G.op_a(A, a_mn), G.op_b(B, b_mn)), **f)
    a = A.t() if a_mn else A
    b = B if b_mn else B.t()
    pre = torch.addmm(f["beta"] * f["C0"] if f["C0"] is not None else torch.zeros(M, N, dtype=torch.float64), a, b,
                      alpha=f["alpha"])
    if f["bias"] is not None:
        pre = pre + f["bias"]
    out = {G.ACT_NONE: pre, G.ACT_RELU: F.relu(pre), G.ACT_SILU: F.silu(pre)}[f["act"]]
    if f["gate"] is not None:
        out = out * (f["gate"] > 0)
    assert torch.allclose(ref["pre"][0], pre, rtol=1e-12, atol=1e-12)
    assert torch.allclose(ref["out"][0], out, rtol=1e-12, atol=1e-12)
    S = f["alpha"] * (a.abs() @ b.abs()) + (abs(f["beta"]) * f["C0"].abs() if f["C0"] is not None else 0)
    S = S + (f["bias"].abs() if f["bias"] is not None else 0)
    assert torch.allclose(ref["pre"][1], S, rtol=1e-12)


EMU_CASES = [  # (M, N, K, layout, splits)
    (200, 96, 1000, "KK", 1),
    (130, 70, 40, "MK", 1),          # one ragged K block
    (64, 160, 616, "KM", 4),         # 10 K blocks in 4 slices
    (50, 40, 560, "MM", 3),          # 9 K blocks in 3 slices
    (16, 64, 8192, "KK", 8),         # the deepest K of the table, split like the skinny kernel's 8 K slabs
]


@pytest.mark.parametrize("M,N,K,layout,splits", EMU_CASES)
def test_emulated_kernel_passes_and_controls_fail(M, N, K, layout, splits):
    a_mn, b_mn = G.LAYOUTS[layout]
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    A, B = G.make_operands(g, M, N, K, a_mn, b_mn)
    C0, bias, gate = G.make_epilogue_inputs(g, M, N, K)
    P = G.Products(G.op_a(A, a_mn), G.op_b(B, b_mn))
    for name, ep in G.EPILOGUES.items():
        f = _fields(ep, C0, bias, gate)
        pre, out, cb = emulate(A, B, a_mn, b_mn, splits, **f)
        ref = G.reference(P, **f)
        got = {"pre": pre, "out": out, "cb": cb}
        for k, r in ref.items():
            ok, ratio, _ = G.check(got[k], *r[:2], TAU, bf16=len(r) > 2)
            assert ok and ratio < TAU / 4, (name, k, ratio)
        if name != "all":
            continue
        for control in G.CONTROLS:
            bad = G.reference(P, control=control, **f)
            worst = max(G.check(got[k], *bad[k][:2], TAU, bf16=len(bad[k]) > 2)[1] for k in bad)
            assert worst >= 20 * TAU, (control, worst)
        want, scale = ref["cb"][:2]
        ok, ratio, _ = G.check(G.bump_one_ulp(cb, want, scale), want, scale, TAU, bf16=True)
        assert not ok and ratio >= 20 * TAU, ratio


def test_routes_of_the_gpu_table():
    for name, (M, N, K, split_k, ws, places, routes) in G.GEMM_CASES.items():
        for layout, want in routes.items():
            for place in places:
                got = G.tc_route(M, N, K, *G.LAYOUTS[layout], split_k, ws or 0, aligned=place == "vec")
                assert got == want, (name, layout, place, got, want)
    for name, (M, N, K, want) in G.SGEMM_CASES.items():
        assert G.sgemm_route(M, N, K) == want, name
    assert G.ops_bf16_route(64, 64, 1000) == "f32" and G.ops_bf16_route(512, 384, 256) == "tc"
    # skinny conditions the table does not reach: N % 4, M > 128, an explicit split_k; the 2^24 cut-off of ops.gemm
    assert G.tc_route(64, 2050, 2048, 0, 0, 0, G.WS_BIG)[0] == 0
    assert G.tc_route(129, 2048, 2048, 0, 0, 0, G.WS_BIG) == (0, 128, 5, 145)      # 32 tiles: automatic split-K
    assert G.tc_route(64, 2048, 2048, 0, 0, 4, G.WS_BIG)[:3] == (0, 128, 4)     # explicit split_k: never skinny
    assert G.ops_bf16_route(64, 64, 4096) == "tc" and G.ops_bf16_route(64, 64, 4095) == "f32"


def test_route_rules_at_their_edges():
    # automatic split-K needs a workspace, fewer than 74 tiles and at least 8 K blocks
    assert G.tc_route(200, 256, 4096, 0, 0, 0, 0)[2] == 1
    assert G.tc_route(200, 256, 448, 0, 0, 0, G.WS_BIG)[2] == 1
    assert G.tc_route(200, 256, 512, 0, 0, 0, G.WS_BIG)[2] == 2
    assert G.tc_route(128 * 74, 128, 4096, 0, 0, 0, G.WS_BIG)[2] == 1
    # explicit split_k is capped by the K blocks, then by the workspace
    assert G.tc_route(100, 100, 128, 0, 0, 8, G.WS_BIG)[2] == 2
    assert G.tc_route(100, 100, 4096, 0, 0, 8, 100 * 100 * 4)[2] == 1
    # the skinny kernel's shared-memory limit at NT = 144: 6 K slabs of 34 KB fit, 7 do not
    assert G.skinny_fits(128, 2048, 3072) == (144, 15) and G.skinny_fits(128, 2048, 3584) is None
