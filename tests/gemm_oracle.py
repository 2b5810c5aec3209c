"""fp64 oracle of the GEMM family (gemm_tc.cu: gemm_tc_kernel, tc_splitk_reduce_kernel, skinny_cluster_kernel;
gemm_f32.cu: sgemm_kernel, splitk_reduce_kernel) and a Python copy of its run-time dispatch rules.

Per output element, in the kernels' order:
  pre = alpha * op(A) op(B) + beta * C0 + bias        (C0 is not read when beta == 0)  -> Cpre
  out = act(pre)                                      (none, ReLU or SiLU)
  out = 0 where gate <= 0                             (0.0 and -0.0 gate too)         -> C
  Cb  = bf16 round-to-nearest-even of out                                             -> Cb
op(A) is M x K (A stored [K][M] when a_mn), op(B) is K x N (B stored [N][K] unless b_mn).  The operands are taken as
given: bf16 tensor-core operands are exact in fp64, so the only error left in a kernel output is its fp32 arithmetic.

Scale of an element: S = |alpha| (|op(A)| |op(B)|) + |beta C0| + |bias|, the first-order bound of the fp32 evaluation
error of pre, which ReLU, SiLU (Lipschitz <= 1.1) and the gate do not enlarge.  The bar is |got - want| <= TAU * S per
element, plus half a bf16 ulp of want on Cb.  TAU comes from fp32 accumulation of exact products: each of the K / 16
MMA steps (or K FMAs) and each split-K / cluster partial adds at most one fp32 rounding of a partial sum bounded by S,
and on random-sign data the partial sums stay orders of magnitude below S, so TAU = 1e-5 (about 170 fp32 unit
roundoffs) leaves room for every kernel's summation order while every control below misses it by far.
Calibration (B200, tests/test_gpu_gemm_oracle.py): the worst kernel error is TAU / 12, the weakest control 53 TAU.

`control` alters the oracle the way a subtle kernel bug would (the tests assert that the check then fails by at least
20 * TAU); `bump_one_ulp` (one bf16 ulp on one element of Cb) alters the kernel output instead:
  "drop_last_kblock"  the last 64-wide K block left out of the product (a split-K slice or ragged K tile lost);
  "transpose_b"       op(B) read in the other layout: the K x N matrix whose row-major elements are op(B)^T's;
  "bias_shift"        the bias of column c - 1 added to column c;
  "ignore_beta"       beta * C0 left out;
  "act_before_bias"   act(alpha A B + beta C0) + bias instead of act(alpha A B + beta C0 + bias).
"""
import torch

from tests.encoder_bf16_oracle import bump_one_ulp, check, ulp_bf16  # noqa: F401  (re-exported for the tests)

TAU = 1e-5
CONTROLS = ("drop_last_kblock", "transpose_b", "bias_shift", "ignore_beta", "act_before_bias")
ACT_NONE, ACT_RELU, ACT_SILU = 0, 1, 2
TC_MACS = 1 << 24            # gemm_tc_from_f32: tensor cores from M * N * K >= 2^24 multiply-adds
BK = 64                      # K block of the tensor-core kernels


def rne(t):
    """The bf16 value the kernels feed the tensor cores (round to nearest even), as float64."""
    return t.float().bfloat16().double()


def op_a(A, a_mn):
    """op(A), M x K, as float64: A stored [K][M] when a_mn, else [M][K]."""
    A = A.double()
    return A.t() if a_mn else A


def op_b(B, b_mn):
    """op(B), K x N, as float64: B stored [K][N] when b_mn, else [N][K]."""
    B = B.double()
    return B if b_mn else B.t()


def act_fn(act, x):
    if act == ACT_RELU:
        return torch.relu(x)
    if act == ACT_SILU:
        return x / (1 + torch.exp(-x))
    return x


class Products:
    """op(A) op(B) and |op(A)| |op(B)| of one operand pair (float64), shared by every epilogue of a case."""

    def __init__(self, a, b):
        self.a, self.b = a, b
        self.ab = a @ b
        self.abs = a.abs() @ b.abs()

    def control(self, control):
        a, b = self.a, self.b
        K, N = b.shape
        if control == "drop_last_kblock":
            k = (K - 1) // BK * BK
            return a[:, :k] @ b[:k]
        if control == "transpose_b":
            return a @ b.t().contiguous().reshape(K, N)
        return self.ab


def reference(P, alpha=1.0, beta=0.0, C0=None, bias=None, act=ACT_NONE, gate=None, control=None):
    """P: Products.  Returns {"pre": (want, S), "out": (want, S), "cb": (want, S, True)} as float64 M x N."""
    ab = P.control(control)
    pre = alpha * ab
    S = abs(alpha) * P.abs
    if beta != 0:
        bc = beta * C0.double()
        S = S + bc.abs()
        if control != "ignore_beta":
            pre = pre + bc
    if bias is not None:
        bv = bias.double()
        S = S + bv.abs()
        if control == "bias_shift":
            bv = torch.roll(bv, 1)
        if control == "act_before_bias":
            out = act_fn(act, pre) + bv
        pre = pre + bv
    if control != "act_before_bias" or bias is None:
        out = act_fn(act, pre)
    if gate is not None:
        out = torch.where(gate.double() <= 0, torch.zeros_like(out), out)
    return {"pre": (pre, S), "out": (out, S), "cb": (out, S, True)}


# ------------------------------------------------------------------------------------------ dispatch rules
def cdiv(a, b):
    return -(-a // b)


def skinny_fits(M, N, K, aligned=True):
    """launch_skinny_cluster's shape and alignment checks; returns (NT, tiles) or None when it declines."""
    if M < 1 or M > 128 or K % (BK * 8) or N % 4 or not aligned:
        return None
    Mpad, kb = (M + 15) // 16 * 16, K // (BK * 8)
    NT = 16 * cdiv(N, 16 * 15)
    if NT > 256 or kb > 8 or (Mpad // 8) * (NT // 4) > 2 * 512:
        return None
    stage = 128 * 128 + (NT * 128 + 1023) // 1024 * 1024
    s_bytes = (Mpad * (NT + 4) * 4 + 1023) // 1024 * 1024
    if max(kb * stage, s_bytes) + 9 * 8 + 16 + 1024 > 227 * 1024:
        return None
    return NT, cdiv(N, NT)


def tc_route(M, N, K, a_mn, b_mn, split_k=0, ws_bytes=0, aligned=True):
    """gemm_tc_bf16's choice: (0 tiled | 1 skinny, BN | NT, z-slices, CTAs), as tacorl_gemm_tc_debug reports it.
    ws_bytes = 0: no workspace; aligned: every output, the gate and the bias pass the skinny kernel's 16-byte checks."""
    BN = 32 if N <= 32 else (64 if N <= 64 else 128)
    skinny = M <= 128 and N >= 512 and K <= 8192 and split_k == 0
    if skinny:
        BN = 64 if b_mn else 32
    if b_mn and BN < 64:
        BN = 64
    if skinny and not a_mn and not b_mn:
        fit = skinny_fits(M, N, K, aligned)
        if fit:
            return (1, fit[0], 8, 8 * fit[1])
    tiles = cdiv(M, 128) * cdiv(N, BN)
    total_kb = cdiv(K, BK)
    splits = split_k
    if splits <= 0:
        splits = 1
        if ws_bytes and not skinny and tiles < 74 and total_kb >= 8:
            splits = min(cdiv(148, tiles), total_kb // 4)
    splits = min(splits, total_kb)
    if splits > 1 and splits * M * N * 4 > ws_bytes:
        splits = max(1, ws_bytes // (M * N * 4))
    per = cdiv(total_kb, splits)
    zs = cdiv(total_kb, per)
    ctas = min(tiles, max(1, 148 // zs))
    return (0, BN, zs, ctas * zs)


def sgemm_route(M, N, K, split_k=0, ws_bytes=96 << 20):
    """gemm_f32's choice: (BM, BN, BK, splits); it launches 1 + (splits > 1) kernels."""
    BM, BN = (256, 32) if N <= 32 else ((128, 64) if N <= 64 else (128, 128))
    ctas = cdiv(M, BM) * cdiv(N, BN)
    small = ctas < 148
    if small:
        BM = BN = 64
        ctas = cdiv(M, 64) * cdiv(N, 64)
    splits = split_k
    if splits <= 0:
        splits = 1
        if ws_bytes and small and K >= 128:
            splits = max(1, min(cdiv(296, ctas), cdiv(K, 64)))
    if splits > 1 and splits * M * N * 4 > ws_bytes:
        splits = ws_bytes // (M * N * 4) if ws_bytes >= 2 * M * N * 4 else 1
    return (BM, BN, 64 if small else 16, splits)


def ops_bf16_route(M, N, K):
    """gemm_tc_from_f32: "f32" (gemm_f32) below 2^24 multiply-adds, else "tc"."""
    return "f32" if M * N * K < TC_MACS else "tc"


# ------------------------------------------------------------------------------------------ the GPU table
# Layouts (a_mn, b_mn): "KK" = both K-major (x W^T), "MK" = A stored [K][M] (dW = dZ^T X), "KM" = B stored [K][N]
# (dX = dZ W), "MM" = both MN-major.
LAYOUTS = {"KK": (0, 0), "MK": (1, 0), "KM": (0, 1), "MM": (1, 1)}
WS_BIG = 64 << 20

# name: (M, N, K, split_k, workspace bytes (None: no workspace), output placements, {layout: route})
# placements: "vec" = 16-byte aligned outputs with pitches that are multiples of 8 (vector epilogue), "scalar" = outputs
# one element off alignment with odd pitches (scalar epilogue).  Both are windows of wider NaN-filled buffers.
_T = lambda r32, r64: {"KK": r32, "MK": r32, "KM": r64, "MM": r64}        # noqa: E731
_ALL = lambda r: {k: r for k in LAYOUTS}                                   # noqa: E731
GEMM_CASES = {
    # tiled kernel (no workspace: no split-K); the debug entry has no 2^24-MAC cut-off
    "tiled_bn32_k8": (3000, 24, 200, 0, None, ("vec", "scalar"), _T((0, 32, 1, 24), (0, 64, 1, 24))),
    "tiled_bn64": (1000, 50, 1000, 0, None, ("vec", "scalar"), _ALL((0, 64, 1, 8))),
    "tiled_bn128_k40": (2570, 1300, 40, 0, None, ("vec", "scalar"), _ALL((0, 128, 1, 148))),
    "tiled_rounds": (5000, 576, 64, 0, None, ("vec", "scalar"), _ALL((0, 128, 1, 148))),
    "tiled_n32_bmn_bn64": (640, 32, 520, 0, None, ("vec", "scalar"), _T((0, 32, 1, 5), (0, 64, 1, 5))),
    # split-K: automatic, explicit (10 K blocks -> 4 slices, 9 K blocks -> 3 of 4), cut to the workspace (8 -> 3)
    "splitk_auto": (200, 256, 4096, 0, WS_BIG, ("vec", "scalar"), _ALL((0, 128, 16, 64))),
    "splitk_10kb_by4": (300, 200, 616, 4, WS_BIG, ("vec", "scalar"), _ALL((0, 128, 4, 24))),
    "splitk_9kb_by4": (300, 200, 560, 4, WS_BIG, ("vec", "scalar"), _ALL((0, 128, 3, 18))),
    "splitk_ws_cut": (260, 130, 1000, 8, 3 * 260 * 130 * 4, ("vec", "scalar"), _ALL((0, 128, 3, 18))),
    # skinny cluster kernel (both operands K-major); the other layouts take the tiled kernel at the skinny BN
    "skinny_64": (64, 2048, 2048, 0, WS_BIG, ("vec",), {"KK": (1, 144, 8, 120), "MK": (0, 32, 1, 64),
                                                        "KM": (0, 64, 1, 32), "MM": (0, 64, 1, 32)}),
    "skinny_ragged_n516": (9, 516, 1024, 0, WS_BIG, ("vec",), {"KK": (1, 48, 8, 88), "MK": (0, 32, 1, 17),
                                                               "KM": (0, 64, 1, 9), "MM": (0, 64, 1, 9)}),
    "skinny_128": (128, 2048, 2048, 0, WS_BIG, ("vec",), {"KK": (1, 144, 8, 120), "MK": (0, 32, 1, 64),
                                                          "KM": (0, 64, 1, 32), "MM": (0, 64, 1, 32)}),
    # skinny shapes the cluster kernel declines: the tiled kernel runs, without split-K
    "skinny_fb_k_not_512": (64, 576, 5000, 0, WS_BIG, ("vec",), {"KK": (0, 32, 1, 18)}),
    "skinny_fb_nt_over_256": (128, 4096, 4096, 0, WS_BIG, ("vec",), {"KK": (0, 32, 1, 128)}),
    "skinny_fb_kslabs_over_8": (100, 1024, 8192, 0, WS_BIG, ("vec",), {"KK": (0, 32, 1, 32)}),
    "skinny_fb_smem": (128, 2048, 4096, 0, WS_BIG, ("vec",), {"KK": (0, 32, 1, 64)}),
    "skinny_fb_unaligned_c": (64, 2048, 2048, 0, WS_BIG, ("scalar",), {"KK": (0, 32, 1, 64)}),
}

# Epilogues: name -> fields.  "c": the fp32 output is written; beta != 0 reads C0 from it, beta == 0 starts it NaN.
EPILOGUES = {
    "none": dict(c=True),
    "bias": dict(c=True, bias=True),
    "beta": dict(c=True, alpha=0.5, beta=0.75),
    "relu": dict(c=True, bias=True, act=ACT_RELU),
    "silu": dict(c=True, bias=True, act=ACT_SILU),
    "cpre": dict(c=True, bias=True, beta=0.75, act=ACT_RELU, cpre=True),
    "gate": dict(c=True, bias=True, act=ACT_RELU, gate=True),
    "cb_only": dict(c=False, cb=True, bias=True, act=ACT_SILU),
    "cb_c": dict(c=True, cb=True, bias=True, beta=0.75, act=ACT_RELU),
    "all": dict(c=True, cb=True, alpha=0.5, beta=0.75, bias=True, act=ACT_SILU, cpre=True, gate=True),
}

# ops.gemm at fp32 precision (gemm_f32): name -> (M, N, K, (BM, BN, BK, splits)) with the automatic split-K
SGEMM_CASES = {
    "sgemm_256x32": (38000, 20, 40, (256, 32, 16, 1)),
    "sgemm_128x64": (19000, 50, 30, (128, 64, 16, 1)),
    "sgemm_128x128": (2000, 1300, 20, (128, 128, 16, 1)),
    "sgemm_64x64_deep": (300, 200, 100, (64, 64, 64, 1)),
    "sgemm_64x64_splitk": (64, 64, 1000, (64, 64, 64, 16)),
}


def make_operands(g, M, N, K, a_mn, b_mn):
    """bf16-exact fp32 operands as stored (values only, dense)."""
    A = torch.randn((K, M) if a_mn else (M, K), generator=g).bfloat16().float()
    B = torch.randn((K, N) if b_mn else (N, K), generator=g).bfloat16().float()
    return A, B


def make_epilogue_inputs(g, M, N, K):
    """C0 and bias at the size of the product (|A B| ~ sqrt(K)), so that the beta and bias controls are visible, and a
    gate with zeros, negative zeros and negatives."""
    C0 = torch.randn(M, N, generator=g) * K ** 0.5
    bias = torch.randn(N, generator=g) * K ** 0.5 / 2
    gate = torch.randn(M, N, generator=g)
    r = torch.rand(M, N, generator=g)
    gate[r < 0.125] = 0.0
    gate[(r >= 0.125) & (r < 0.25)] = -0.0
    return C0, bias, gate
