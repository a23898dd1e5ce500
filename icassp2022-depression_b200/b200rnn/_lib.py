"""ctypes binding of the C-ABI library (include/b200rnn.h).

There is no CPU fallback by design: if ``lib/libb200rnn.so`` is missing or does not export the symbols the
header declares, importing the compute entry points fails loudly.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_uint32, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200RNN_LIB: load another build of the SAME library (e.g. the -DB200RNN_TRACE build used by tools/trace_rec.py)
LIB_PATH = os.environ.get("B200RNN_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libb200rnn.so")

GRU, LSTM = 0, 1
FLAG_ACCUMULATE_GRADS = 1
FLAG_SAVE_FOR_BACKWARD = 2
FLAG_FUSED_LN = 4
ABI_VERSION = 2

# every symbol include/b200rnn.h declares (tests check the .so exports exactly these)
SYMBOLS = (
    "b200rnn_version",
    "b200rnn_last_error",
    "b200rnn_sm_count",
    "b200rnn_launch_count",
    "b200rnn_workspace_bytes",
    "b200rnn_forward",
    "b200rnn_forward_fused",
    "b200rnn_backward",
    "b200rnn_backward_fused",
    "b200rnn_wcache_bytes",
    "b200rnn_prepare_weights",
    "b200rnn_gemm_f32",
    "b200rnn_attention_pool",
    "b200rnn_attention_pool_bwd",
    "b200rnn_mlp_dropout",
    "b200rnn_rng_next",
    "b200rnn_fuse_loss_grad",
    "b200rnn_softmax_ce",
    "b200rnn_adam",
    "b200rnn_adamw",
    "b200rnn_fuse_head",
    "b200rnn_fuse_head_finish",
    "b200rnn_fuse_head_scratch_floats",
    "b200rnn_comm_bytes",
    "b200rnn_comm_create",
    "b200rnn_comm_open",
    "b200rnn_comm_close",
    "b200rnn_comm_destroy",
    "b200rnn_profile",
    "b200rnn_profile_read",
)
COMM_MAX_WORLD = 8
IPC_HANDLE_BYTES = 64


class Desc(ctypes.Structure):
    """``b200rnn_desc`` (include/b200rnn.h)."""

    _fields_ = [
        ("mode", c_int32),
        ("batch", c_int32),
        ("seq_len", c_int32),
        ("input_size", c_int32),
        ("hidden_size", c_int32),
        ("num_layers", c_int32),
        ("num_dirs", c_int32),
        ("training", c_int32),
        ("dropout_p", c_float),
        ("flags", c_uint32),
    ]


class FuseHeadArgs(ctypes.Structure):
    """``b200rnn_fuse_head_args`` (include/b200rnn.h), field for field."""

    _fields_ = [
        ("struct_bytes", c_uint32),
        ("B", c_int32), ("T", c_int32), ("Ht", c_int32), ("Ha", c_int32),
        ("n_states", c_int32),
        ("training", c_int32),
        ("p", c_float),
        ("regression", c_int32),
        ("accumulate", c_int32),
        ("do_adam", c_int32),
        ("world", c_int32), ("rank", c_int32), ("defer_exchange", c_int32),
        ("lr", c_float), ("beta1", c_float), ("beta2", c_float), ("eps", c_float), ("grad_scale", c_float),
        ("rng_consume", c_uint64),
        ("seq_st", c_int64), ("seq_sb", c_int64),
        ("seq", c_void_p), ("h_n", c_void_p), ("w_att", c_void_p), ("b_att", c_void_p),
        ("ctx_in", c_void_p), ("ctx_out", c_void_p), ("tf_in", c_void_p),
        ("w_t", c_void_p), ("b_t", c_void_p), ("pooled", c_void_p), ("w_a", c_void_p), ("b_a", c_void_p),
        ("rng_state", c_void_p),
        ("text_feature", c_void_p), ("audio_feature", c_void_p),
        ("W", c_void_p), ("w_modal", c_void_p), ("labels", c_void_p),
        ("out", c_void_p), ("loss", c_void_p), ("dw_part", c_void_p), ("dw", c_void_p), ("ticket", c_void_p),
        ("adam_m", c_void_p), ("adam_v", c_void_p), ("adam_step", c_void_p),
        ("comm_step", c_void_p), ("comm_done", c_void_p),
        ("comm_buf", c_void_p * 8),
    ]

    def __init__(self, **kw):
        super().__init__(**kw)
        self.struct_bytes = ctypes.sizeof(FuseHeadArgs)


class B200RNNError(RuntimeError):
    pass


_lib = None


def load() -> ctypes.CDLL:
    """Load (once) and type the shared library. Raises if it is absent — no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200RNNError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C icassp2022-depression_b200`). b200rnn has no CPU / PyTorch fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    missing = [s for s in SYMBOLS if not hasattr(lib, s)]
    if missing:
        raise B200RNNError(f"{LIB_PATH} does not export {missing}")
    fp = POINTER(c_float)
    lib.b200rnn_version.restype = c_int
    lib.b200rnn_version.argtypes = []
    lib.b200rnn_last_error.restype = c_char_p
    lib.b200rnn_last_error.argtypes = []
    lib.b200rnn_launch_count.restype = ctypes.c_ulonglong
    lib.b200rnn_launch_count.argtypes = []
    lib.b200rnn_sm_count.restype = c_int
    lib.b200rnn_sm_count.argtypes = []
    lib.b200rnn_workspace_bytes.restype = c_int
    lib.b200rnn_workspace_bytes.argtypes = [POINTER(Desc), POINTER(c_size_t), POINTER(c_size_t)]
    lib.b200rnn_forward.restype = c_int
    lib.b200rnn_forward.argtypes = [
        POINTER(Desc), c_void_p, c_int64, c_int64,  # desc, x, strides
        POINTER(c_void_p),                           # params
        c_void_p, c_int64, c_int64,                  # y, strides
        c_void_p, c_void_p,                          # h_n, c_n
        c_void_p, c_void_p,                          # reserve, scratch
        c_uint64, c_uint64, c_void_p,                # seed, offset, rng_state
        c_void_p,                                    # stream
    ]
    lib.b200rnn_forward_fused.restype = c_int
    lib.b200rnn_forward_fused.argtypes = lib.b200rnn_forward.argtypes[:-1] + [c_void_p, c_void_p, c_float, c_void_p,
                                                                              c_void_p, c_void_p, c_void_p]
    lib.b200rnn_wcache_bytes.restype = c_int
    lib.b200rnn_wcache_bytes.argtypes = [POINTER(Desc), POINTER(c_size_t)]
    lib.b200rnn_prepare_weights.restype = c_int
    lib.b200rnn_prepare_weights.argtypes = [POINTER(Desc), POINTER(c_void_p), c_void_p, c_void_p]
    lib.b200rnn_backward.restype = c_int
    lib.b200rnn_backward.argtypes = [
        POINTER(Desc), c_void_p, c_int64, c_int64,   # desc, x, strides
        POINTER(c_void_p),                           # params
        c_void_p, c_int64, c_int64,                  # y
        c_void_p, c_int64, c_int64,                  # dy
        c_void_p, c_void_p,                          # dh_n, dc_n
        c_void_p, c_void_p,                          # reserve, scratch
        c_void_p, c_int64, c_int64,                  # dx
        POINTER(c_void_p),                           # dparams
        c_void_p,                                    # lengths
        c_void_p,                                    # stream
    ]
    lib.b200rnn_backward_fused.restype = c_int
    lib.b200rnn_backward_fused.argtypes = [
        POINTER(Desc), c_void_p, c_int64, c_int64,   # desc, x, strides
        POINTER(c_void_p),                           # params
        c_void_p, c_int64, c_int64,                  # y
        c_void_p, c_int64, c_int64,                  # dy
        c_void_p, c_float,                           # dy_pool, dy_pool_scale
        c_void_p, c_void_p,                          # dh_n, dc_n
        c_void_p, c_void_p,                          # reserve, scratch
        c_void_p, c_int64, c_int64,                  # dx
        POINTER(c_void_p),                           # dparams
        c_void_p,                                    # lengths
        c_void_p, c_float, c_void_p, c_void_p,       # ln_gamma, ln_eps, dln_gamma, dln_beta
        c_void_p,                                    # stream
    ]
    lib.b200rnn_gemm_f32.restype = c_int
    lib.b200rnn_gemm_f32.argtypes = [
        c_int, c_int, c_int, c_void_p, c_int64, c_int, c_void_p, c_int64, c_int, c_void_p, c_int64, c_void_p,
        c_int, c_void_p, c_size_t, c_void_p,
    ]
    lib.b200rnn_attention_pool.restype = c_int
    lib.b200rnn_attention_pool.argtypes = [c_void_p, c_int64, c_int64, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                           c_void_p, c_void_p, c_void_p]
    lib.b200rnn_attention_pool_bwd.restype = c_int
    lib.b200rnn_attention_pool_bwd.argtypes = [c_void_p, c_int64, c_int64, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                               c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p,
                                               c_void_p, c_void_p]
    lib.b200rnn_mlp_dropout.restype = c_int
    lib.b200rnn_mlp_dropout.argtypes = [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_float, c_void_p,
                                        c_uint32, c_void_p]
    lib.b200rnn_rng_next.restype = c_int
    lib.b200rnn_rng_next.argtypes = [c_void_p, c_void_p, c_uint64, c_void_p]
    lib.b200rnn_fuse_loss_grad.restype = c_int
    lib.b200rnn_fuse_loss_grad.argtypes = [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                           c_void_p, c_void_p, c_void_p]
    lib.b200rnn_softmax_ce.restype = c_int
    lib.b200rnn_softmax_ce.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.b200rnn_adam.restype = c_int
    lib.b200rnn_adam.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_float,
                                 c_float, c_void_p]
    lib.b200rnn_adamw.restype = c_int
    lib.b200rnn_adamw.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_float,
                                  c_float, c_float, c_float, c_int, c_void_p]
    lib.b200rnn_fuse_head.restype = c_int
    lib.b200rnn_fuse_head.argtypes = [POINTER(FuseHeadArgs), c_void_p]
    lib.b200rnn_fuse_head_finish.restype = c_int
    lib.b200rnn_fuse_head_finish.argtypes = [POINTER(FuseHeadArgs), c_void_p]
    lib.b200rnn_fuse_head_scratch_floats.restype = c_size_t
    lib.b200rnn_fuse_head_scratch_floats.argtypes = [c_int, c_int, c_int, c_int]
    lib.b200rnn_comm_bytes.restype = c_size_t
    lib.b200rnn_comm_bytes.argtypes = []
    lib.b200rnn_comm_create.restype = c_int
    lib.b200rnn_comm_create.argtypes = [POINTER(c_void_p), POINTER(ctypes.c_ubyte)]
    lib.b200rnn_comm_open.restype = c_int
    lib.b200rnn_comm_open.argtypes = [POINTER(ctypes.c_ubyte), POINTER(c_void_p)]
    lib.b200rnn_comm_close.restype = c_int
    lib.b200rnn_comm_close.argtypes = [c_void_p]
    lib.b200rnn_comm_destroy.restype = c_int
    lib.b200rnn_comm_destroy.argtypes = [c_void_p]
    lib.b200rnn_profile.restype = c_int
    lib.b200rnn_profile.argtypes = [c_int]
    lib.b200rnn_profile_read.restype = c_int
    lib.b200rnn_profile_read.argtypes = [c_int, POINTER(c_float), POINTER(c_int)]
    del fp
    v = lib.b200rnn_version()
    if v != ABI_VERSION:
        raise B200RNNError(f"ABI mismatch: library {v}, binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().b200rnn_last_error().decode("utf-8", "replace")
        raise B200RNNError(f"{what} failed (code {rc}): {msg}")


def workspace_bytes(desc: Desc) -> tuple[int, int]:
    r, s = c_size_t(0), c_size_t(0)
    check(load().b200rnn_workspace_bytes(ctypes.byref(desc), ctypes.byref(r), ctypes.byref(s)), "workspace_bytes")
    return int(r.value), int(s.value)


def ptr_array(ptrs) -> ctypes.Array:
    arr = (c_void_p * len(ptrs))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr


PROF_REC_FWD, PROF_REC_BWD, PROF_GEMM, PROF_MISC = 0, 1, 2, 3


def profile(enable: bool) -> None:
    check(load().b200rnn_profile(1 if enable else 0), "profile")


def profile_read(kind: int) -> tuple[float, int]:
    """(total milliseconds, launches) of the library's launches of ``kind`` since profiling was enabled."""
    ms, n = c_float(0.0), c_int(0)
    check(load().b200rnn_profile_read(kind, ctypes.byref(ms), ctypes.byref(n)), "profile_read")
    return float(ms.value), int(n.value)


def launch_count() -> int:
    return int(load().b200rnn_launch_count())
