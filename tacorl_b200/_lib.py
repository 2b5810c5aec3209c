"""ctypes binding of the C-ABI library (include/tacorl_b200.h).

There is NO fallback: if `lib/libtacorl_b200.so` is missing or a call is made on non-CUDA
tensors this raises.  Build with `python tacorl_b200/csrc/build.py` (or __graft_entry__.build()).
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtacorl_b200.so")

PREC_F32, PREC_BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_SILU = 0, 1, 2
ACTS = {None: ACT_NONE, "none": ACT_NONE, "relu": ACT_RELU, "silu": ACT_SILU}

_lib = None

_vp, _i, _ll, _f, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_float, ctypes.c_size_t

# name -> argtypes (restype int unless listed in _RESTYPES)
_SIGS = {
    "tacorl_gemm": [_i, _i, _i, _i, _i, _f, _vp, _ll, _vp, _ll, _f, _vp, _ll, _vp, _i, _vp, _ll, _vp, _sz, _i, _vp],
    "tacorl_gemm_ex": [_i, _i, _i, _i, _i, _f, _vp, _ll, _vp, _ll, _f, _vp, _ll, _vp, _i, _vp, _ll, _vp, _vp, _vp, _sz, _i,
                       _vp],
    "tacorl_colsum": [_i, _i, _vp, _ll, _vp, _i, _vp],
    "tacorl_act_bwd": [_i, _ll, _vp, _vp, _vp, _vp],
    "tacorl_scale": [_ll, _vp, _vp, _f, _vp, _vp],
    "tacorl_rowscale": [_ll, _i, _vp, _vp, _f, _vp, _i, _vp],
    "tacorl_lmp_encoder_ws_bytes": [_i, _i, _i, _i, _i, _i],
    "tacorl_lmp_encoder_fwd": [_vp, _i, _f, _f, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _i, _vp],
    "tacorl_lmp_encoder_bwd": [_vp, _i, _f, _f, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i,
                               _vp, _vp, _sz, _i, _vp],
    "tacorl_conv_tc_debug": [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp],
    "tacorl_rnn_layer_ws_bytes": [_i, _i, _i, _i],
    "tacorl_rnn_layer_fwd": [_i, _i, _i, _i, _vp, _ll, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _ll, _vp, _vp, _vp, _vp, _sz,
                             _i, _vp],
    "tacorl_rnn_layer_bwd": [_i, _i, _i, _i, _vp, _ll, _vp, _vp, _vp, _i, _i, _vp, _ll, _vp, _ll, _vp, _vp, _ll, _i,
                             _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _sz, _i, _vp],
    "tacorl_rnn_layer2_ws_bytes": [_i, _i, _i, _i, _i],
    "tacorl_rnn_layer2_fwd": [_i, _i, _i, _i, _i, _vp, _ll, _vp, _ll, _vp, _vp, _vp, _vp, _ll, _vp, _vp, _sz, _vp],
    "tacorl_rnn_layer2_bwd": [_i, _i, _i, _i, _i, _i, _vp, _ll, _vp, _ll, _vp, _vp, _vp, _vp, _ll, _vp, _vp, _ll, _vp, _vp, _ll,
                              _vp, _vp, _sz, _vp],
    "tacorl_cast_transpose_bf16": [_vp, _i, _i, _vp, _vp],
    "tacorl_dlm_nll": [_i, _i, _vp, _ll, _vp, _ll, _i, _f, _f, _f, _vp, _vp, _vp, _ll, _vp],
    "tacorl_dlm_sample": [_i, _i, _vp, _ll, _vp, _vp, _vp, _ll, _f, _f, _vp, _vp, _vp, _vp],
    "tacorl_gauss_head_fwd": [_i, _i, _vp, _vp, _vp, _vp],
    "tacorl_gauss_head_bwd": [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "tacorl_softplus_head_fwd": [_i, _i, _vp, _f, _vp, _vp, _vp],
    "tacorl_softplus_head_bwd": [_i, _i, _vp, _vp, _vp, _vp, _vp],
    "tacorl_kl_balanced": [_i, _i, _vp, _vp, _vp, _vp, _f, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "tacorl_tanh_rsample_fwd": [_ll, _ll, _vp, _vp, _vp, _vp, _vp, _i, _vp],
    "tacorl_tanh_rsample_bwd": [_ll, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp],
    "tacorl_tanh_logprob": [_i, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp],
    "tacorl_gripper_gumbel": [_i, _i, _vp, _vp, _i, _vp, _vp, _vp],
    "tacorl_gripper_logprob": [_i, _i, _vp, _vp, _vp, _vp],
    "tacorl_gripper_logprob_bwd": [_i, _vp, _vp, _vp, _vp, _vp],
    "tacorl_posemb_fwd": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "tacorl_posemb_bwd": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "tacorl_attn_fwd": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "tacorl_attn_bwd": [_i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "tacorl_add_ln_fwd": [_i, _i, _vp, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp],
    "tacorl_add_ln_bwd": [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tacorl_mean_t_fwd": [_i, _i, _i, _vp, _vp, _vp],
    "tacorl_mean_t_bwd": [_i, _i, _i, _vp, _vp, _vp],
    "tacorl_mul": [_ll, _vp, _vp, _vp, _vp],
    "tacorl_cql_critic_loss": [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _f, _f, _f, _f, _i,
                               _vp, _vp, _vp, _vp, _vp],
    "tacorl_cql_actor_loss": [_i, _i, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp, _vp, _vp],
    "tacorl_dp_unique_id": [_vp],
    "tacorl_dp_allreduce_init": [_vp, _i, _i],
    "tacorl_dp_allreduce_enqueue": [_vp, _ll, _i, _vp],
    "tacorl_dp_allreduce_wait": [_vp],
    "tacorl_dp_allreduce_destroy": [],
    "tacorl_window_gather_u8": [_vp, _ll, _i, _i, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp],
    "tacorl_actions_gather_pad": [_vp, _ll, _i, _vp, _vp, _i, _i, _i, _vp, _vp],
    "tacorl_color_jitter_u8": [_vp, _ll, _i, _i, _vp, _vp, _f, _f, _vp, _vp, _vp],
    "tacorl_replay_sample": [_i, _i, _i, _i, _i, _i, _i, ctypes.c_ulonglong, ctypes.c_ulonglong, _i, _vp, _vp, _ll, _vp,
                             _ll, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "tacorl_replay_gather": [_i, _i, _i, _vp, _i, _vp, _vp, _i, _i, _i, _vp, _vp],
    "tacorl_replay_color_jitter": [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _f, _f, _vp, _vp, _vp],
    "tacorl_replay_sweep": [_i, _i, _i, _i, _i, ctypes.c_ulonglong, ctypes.c_ulonglong, _i, _vp, _vp, _ll, _vp, _ll, _vp,
                            _i, _vp, _vp, _vp],
    "tacorl_replay_gather_rows": [_i, _i, _i, _i, _vp, _i, _vp, _vp, _i, _i, _i, _vp, _vp],
    "tacorl_metrics_accumulate": [_vp, _vp, _vp],
    "tacorl_metrics_record": [_vp, _vp, _i, _vp, _vp, _vp],
    "tacorl_mlp_chain_ws_bytes": [_i, _i, _vp],
    "tacorl_mlp_chain_fwd": [_i, _i, _vp, _vp, _i, _ll, _vp, _i, _ll, _vp, _ll, _vp, _ll, _vp],
    "tacorl_mlp_chain_bwd": [_i, _i, _vp, _vp, _i, _ll, _vp, _i, _ll, _vp, _ll, _vp, _ll, _vp, _ll, _vp, _ll, _vp, _sz, _vp],
    "tacorl_adam_step": [_ll, _vp, _vp, _vp, _vp, _f, _f, _f, _f, _i, _vp, _f, _vp, _f, _vp, _vp],
    "tacorl_adam_step_range": [_ll, _vp, _vp, _vp, _vp, _f, _f, _f, _f, _i, _vp, _i, _i, _f, _vp, _f, _vp, _vp],
    "tacorl_polyak_update": [_ll, _vp, _vp, _f, _vp],
    "tacorl_sqnorm": [_ll, _vp, _vp, _vp, _vp],
    "tacorl_last_error": [],
    "tacorl_abi_version": [],
    "tacorl_launch_count": [],
    "tacorl_rnn_seq_timeouts": [],
    "tacorl_rnn_seq_enable": [_i],
    "tacorl_set_sm_reserve": [_i],
}
_RESTYPES = {
    "tacorl_lmp_encoder_ws_bytes": _sz, "tacorl_rnn_layer_ws_bytes": _sz, "tacorl_rnn_layer2_ws_bytes": _sz,
    "tacorl_mlp_chain_ws_bytes": _sz,
    "tacorl_last_error": ctypes.c_char_p, "tacorl_launch_count": ctypes.c_ulonglong,
    "tacorl_rnn_seq_timeouts": ctypes.c_uint,
}
EXPORTED = tuple(_SIGS)


class TacorlLibraryError(RuntimeError):
    pass


class MlpLayer(ctypes.Structure):
    """tacorl_mlp_layer (include/tacorl_b200.h)."""
    _fields_ = [("W0", _vp), ("b0", _vp), ("n0", _i), ("W1", _vp), ("b1", _vp), ("n1", _i),
                ("W2", _vp), ("b2", _vp), ("n2", _i), ("in_", _i), ("act", _i),
                ("dW0", _vp), ("db0", _vp), ("dW1", _vp), ("db1", _vp), ("dW2", _vp), ("db2", _vp)]


class ReplayImage(ctypes.Structure):
    """tacorl_replay_image (include/tacorl_b200.h)."""
    _fields_ = [("store", _vp), ("out", _vp), ("shift", _vp), ("H", _i), ("W", _i), ("role", _i),
                ("shift_slot", _i), ("n_slots", _i)]


class ReplayJitter(ctypes.Structure):
    """tacorl_replay_jitter (include/tacorl_b200.h)."""
    _fields_ = [("ops", _i), ("lo", _f * 3), ("span", _f * 3)]


REPLAY_WINDOW, REPLAY_OBS, REPLAY_NEXT, REPLAY_GOAL = 0, 1, 2, 3
REPLAY_MAX_IMAGES = 8
METRICS_MAX = 32


class Metrics(ctypes.Structure):
    """tacorl_metrics (include/tacorl_b200.h)."""
    _fields_ = [("value", _vp * METRICS_MAX), ("k", _i), ("n", _i)]


def lib():
    """The loaded shared library.  Fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TacorlLibraryError(
                f"{LIB_PATH} not found: the CUDA extension is not built (run "
                "`python tacorl_b200/csrc/build.py`).  tacorl_b200 has no CPU / eager fallback.")
        L = ctypes.CDLL(LIB_PATH)
        for name, args in _SIGS.items():
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = _RESTYPES.get(name, ctypes.c_int)
        _lib = L
    return _lib


def call(name, *args):
    """Call an int-returning entry point; raise with tacorl_last_error() on failure."""
    L = lib()
    rc = getattr(L, name)(*args)
    if rc != 0:
        raise TacorlLibraryError(f"{name} failed ({rc}): {L.tacorl_last_error().decode()}")


def query(name, *args):
    return getattr(lib(), name)(*args)


def launch_count():
    return int(lib().tacorl_launch_count())


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t, allow_none=True):
    """Device pointer of a contiguous fp32 CUDA tensor (or NULL)."""
    if t is None:
        if allow_none:
            return None
        raise TacorlLibraryError("null tensor")
    if not t.is_cuda:
        raise TacorlLibraryError("tacorl_b200 ops need CUDA tensors (there is no CPU fallback)")
    if t.dtype != torch.float32:
        raise TacorlLibraryError(f"expected float32, got {t.dtype}")
    return ctypes.c_void_p(t.data_ptr())


def ptr_any(t):
    """Device pointer of a contiguous CUDA tensor of any dtype (saved bf16 activations)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise TacorlLibraryError("tacorl_b200 ops need CUDA tensors (there is no CPU fallback)")
    return ctypes.c_void_p(t.data_ptr())


def ptr_array(tensors):
    """void*[] of device pointers (None -> NULL)."""
    arr = (ctypes.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = None if t is None else t.data_ptr()
    return arr


def int_array(values):
    return (ctypes.c_int * len(values))(*[int(v) for v in values])


_WS = {}
# outgrown scratch buffers stay allocated: a CUDA graph captured earlier (a training step) still reads and writes them
# when a larger call (a validation batch bigger than the training batch) has moved on to a new buffer
_WS_RETIRED = []


def workspace(nbytes, device, tag="main"):
    """Cached per-device scratch buffer (stream-ordered reuse on the current stream)."""
    if torch.device(device).type != "cuda":
        raise TacorlLibraryError("tacorl_b200 ops need CUDA tensors (there is no CPU fallback)")
    key = (device.index if device.index is not None else torch.cuda.current_device(), tag)
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        if buf is not None:
            _WS_RETIRED.append(buf)
        buf = torch.empty(int(nbytes * 1.25) + 4096, dtype=torch.uint8, device=device)
        _WS[key] = buf
    return buf
