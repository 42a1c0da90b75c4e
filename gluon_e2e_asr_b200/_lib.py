"""ctypes binding of libctcb.so (include/ctcb.h, include/ctcb_dlpack.h).

The library is built in-tree by ``__graft_entry__.build()``; importing the
compute API without it fails loudly -- there is no Python or CPU fallback for the path.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# CTCB_LIB_PATH: another build of the same library (A/B measurements of kernel changes)
LIB_PATH = os.environ.get("CTCB_LIB_PATH") or os.path.join(_HERE, "libctcb.so")

CTCB_OK, CTCB_INVALID_VALUE, CTCB_WORKSPACE_TOO_SMALL, CTCB_EXECUTION_FAILED, CTCB_MEMOPS_FAILED, CTCB_UNSUPPORTED = range(6)
DT_I32, DT_I64, DT_F32, DT_F64 = range(4)
DT_BF16 = 4             # CTCB_BF16: a logits type only (the *_typed entries), never a label or length type
UTT_INFEASIBLE, UTT_BAD_LABEL, UTT_LEN_CLAMPED, UTT_WIDE_LOGITS = 1, 2, 4, 8
LAYOUT_NTC, LABEL_TN, KEEP_FOR_BACKWARD = 1, 2, 4
PHASE_FUSED, PHASE_FORWARD, PHASE_BACKWARD = 0 << 8, 1 << 8, 2 << 8

EXPORTS = (
    "ctcb_version", "ctcb_last_error", "ctcb_workspace_bytes", "ctcb_loss_grad", "ctcb_forward",
    "ctcb_backward", "ctcb_loss_grad_host", "ctcb_greedy_decode", "ctcb_loss_sum_allreduce",
    "ctcb_last_launch_count", "ctcb_last_walk_config", "ctcb_loss_grad_dlpack", "ctcb_loss_grad_timed",
    "ctcb_scale_rows", "ctcb_edit_distance", "ctcb_loss_grad_host_resident",
    "ctcb_pipe_create", "ctcb_pipe_submit", "ctcb_pipe_wait", "ctcb_pipe_destroy", "ctcb_pipe_last_h2d_bytes",
    "ctcb_mailbox_create", "ctcb_mailbox_handle", "ctcb_mailbox_connect", "ctcb_mailbox_exchange",
    "ctcb_mailbox_flush", "ctcb_mailbox_destroy", "ctcb_mailbox_exchange_with_next",
    "ctcb_set_option", "ctcb_get_option", "ctcb_greedy_decode_unk", "ctcb_last_grad_kernel",
    "ctcb_proj_forward", "ctcb_proj_loss_grad",
    "ctcb_loss_grad_typed", "ctcb_forward_typed", "ctcb_backward_typed", "ctcb_greedy_decode_typed",
    "ctcb_proj_forward_decode", "ctcb_proj_greedy_decode", "ctcb_proj_backward", "ctcb_forward_decode_typed",
)


class CtcbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libctcb error %d: %s" % (code, msg))
        self.code = code


class Problem(ctypes.Structure):
    """ctcb_problem_t (include/ctcb.h)."""
    _fields_ = [
        ("T", ctypes.c_int32), ("B", ctypes.c_int32), ("V", ctypes.c_int32), ("Lmax", ctypes.c_int32),
        ("blank", ctypes.c_int32), ("label_pad", ctypes.c_int32),
        ("logits", ctypes.c_void_p), ("logits_stride_t", ctypes.c_int64), ("logits_stride_b", ctypes.c_int64),
        ("grad", ctypes.c_void_p), ("grad_stride_t", ctypes.c_int64), ("grad_stride_b", ctypes.c_int64),
        ("labels", ctypes.c_void_p), ("label_dtype", ctypes.c_int32),
        ("label_stride_b", ctypes.c_int64), ("label_stride_l", ctypes.c_int64),
        ("data_lengths", ctypes.c_void_p), ("data_lengths_dtype", ctypes.c_int32),
        ("label_lengths", ctypes.c_void_p), ("label_lengths_dtype", ctypes.c_int32),
        ("head_grad", ctypes.c_void_p), ("loss", ctypes.c_void_p), ("loss_sum", ctypes.c_void_p),
        ("status", ctypes.c_void_p), ("logits_row_offsets", ctypes.c_void_p),
    ]


class Proj(ctypes.Structure):
    """ctcb_proj_t (include/ctcb.h): the output projection in front of the loss."""
    _fields_ = [
        ("hidden", ctypes.c_void_p), ("hidden_stride_t", ctypes.c_int64), ("hidden_stride_b", ctypes.c_int64),
        ("K", ctypes.c_int32), ("weight", ctypes.c_void_p), ("bias", ctypes.c_void_p), ("operand_dtype", ctypes.c_int32),
    ]


_lib = None


def load():
    """Returns the loaded library; raises if the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "gluon_e2e_asr_b200: %s is missing -- run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback for the CTC path." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_size_t
    PP = ctypes.POINTER(Problem)
    lib.ctcb_version.restype = ctypes.c_int
    lib.ctcb_last_error.restype = ctypes.c_char_p
    lib.ctcb_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, ctypes.POINTER(sz)]
    lib.ctcb_loss_grad.argtypes = [PP, vp, sz, vp]
    lib.ctcb_forward.argtypes = [PP, i32, vp, sz, vp]
    lib.ctcb_backward.argtypes = [PP, vp, sz, vp]
    lib.ctcb_loss_grad_typed.argtypes = [PP, i32, vp, sz, vp]
    lib.ctcb_forward_typed.argtypes = [PP, i32, i32, vp, sz, vp]
    lib.ctcb_backward_typed.argtypes = [PP, i32, vp, sz, vp]
    lib.ctcb_forward_decode_typed.argtypes = [PP, i32, i32, vp, vp, vp, sz, vp]
    lib.ctcb_loss_grad_timed.argtypes = [PP, vp, sz, vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(i32)]
    lib.ctcb_loss_grad_host.argtypes = [PP, ctypes.c_int]
    lib.ctcb_loss_grad_host_resident.argtypes = [PP, ctypes.c_int, ctypes.POINTER(vp)]
    lib.ctcb_pipe_create.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.POINTER(vp)]
    lib.ctcb_pipe_submit.argtypes = [vp, PP, ctypes.POINTER(i64)]
    lib.ctcb_pipe_wait.argtypes = [vp, i64, ctypes.POINTER(vp)]
    lib.ctcb_pipe_destroy.argtypes = [vp]
    lib.ctcb_pipe_last_h2d_bytes.argtypes = [vp, ctypes.POINTER(i64), ctypes.POINTER(i32)]
    lib.ctcb_mailbox_create.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(vp)]
    lib.ctcb_mailbox_handle.argtypes = [vp, vp]
    lib.ctcb_mailbox_connect.argtypes = [vp, vp]
    lib.ctcb_mailbox_exchange.argtypes = [vp, vp, i32, vp, vp]
    lib.ctcb_mailbox_flush.argtypes = [vp, i32, vp, vp]
    lib.ctcb_mailbox_exchange_with_next.argtypes = [vp, vp, i32, vp]
    lib.ctcb_mailbox_destroy.argtypes = [vp]
    lib.ctcb_greedy_decode.argtypes = [vp, i64, i64, vp, i32, i32, i32, i32, i32, vp, vp, vp]
    lib.ctcb_greedy_decode_unk.argtypes = [vp, i64, i64, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp]
    lib.ctcb_greedy_decode_typed.argtypes = [vp, i32, i64, i64, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp]
    lib.ctcb_scale_rows.argtypes = [vp, i64, i64, i32, i32, i32, vp, vp]
    lib.ctcb_edit_distance.argtypes = [vp, i64, vp, vp, i64, vp, i32, i32, i32, vp, vp, vp]
    lib.ctcb_loss_sum_allreduce.argtypes = [vp, vp, i32, vp]
    lib.ctcb_last_walk_config.argtypes = [ctypes.POINTER(i32), ctypes.POINTER(i32)]
    lib.ctcb_loss_grad_dlpack.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, sz, vp]
    lib.ctcb_proj_forward.argtypes = [ctypes.POINTER(Proj), PP, i32, vp, sz, vp]
    lib.ctcb_proj_loss_grad.argtypes = [ctypes.POINTER(Proj), PP, vp, sz, vp]
    lib.ctcb_proj_backward.argtypes = [ctypes.POINTER(Proj), PP, vp, sz, vp]
    lib.ctcb_proj_forward_decode.argtypes = [ctypes.POINTER(Proj), PP, i32, i32, vp, vp, vp, sz, vp]
    lib.ctcb_proj_greedy_decode.argtypes = [ctypes.POINTER(Proj), i32, i32, i32, vp, i32, i32, i32, vp, vp, vp]
    lib.ctcb_set_option.argtypes = [ctypes.c_char_p, i32]
    lib.ctcb_get_option.argtypes = [ctypes.c_char_p, ctypes.POINTER(i32)]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name != "ctcb_last_error":
            fn.restype = ctypes.c_int
    _lib = lib
    return lib


def check(rc):
    if rc != CTCB_OK:
        raise CtcbError(rc, load().ctcb_last_error().decode("utf-8", "replace"))


_ws_bytes = {}
_opt_epoch = 0          # bumped by set_option: cached workspace sizes depend on walk_p / walk_nw / fused


def set_option(name, value):
    """ctcb_set_option: tuning / experiment switch (tests, A/B runs); -1 = automatic."""
    global _opt_epoch
    check(load().ctcb_set_option(name.encode(), int(value)))
    _opt_epoch += 1


def get_option(name):
    v = ctypes.c_int32(0)
    check(load().ctcb_get_option(name.encode(), ctypes.byref(v)))
    return int(v.value)


class options:
    """``with options(overlap=0, fused=0): ...`` -- sets the switches, restores the previous values."""

    def __init__(self, **kw):
        self.kw, self.old = kw, {}

    def __enter__(self):
        for k, v in self.kw.items():
            self.old[k] = get_option(k)
            set_option(k, v)
        return self

    def __exit__(self, *exc):
        for k, v in self.old.items():
            set_option(k, v)
        return False


def workspace_bytes(T, B, V, Lmax, need_grad=True):
    key = (T, B, V, Lmax, bool(need_grad), _opt_epoch)
    n = _ws_bytes.get(key)
    if n is None:
        out = ctypes.c_size_t(0)
        check(load().ctcb_workspace_bytes(T, B, V, Lmax, 1 if need_grad else 0, ctypes.byref(out)))
        n = _ws_bytes[key] = out.value
    return n


def last_launch_count():
    return int(load().ctcb_last_launch_count())


def last_grad_kernel():
    """Name of the gradient kernel the last call on this thread launched (ctcb_last_grad_kernel)."""
    return {0: None, 1: "k_grad", 2: "k_grad2", 3: "k_meet"}[int(load().ctcb_last_grad_kernel())]


def last_walk_config():
    p, nw = ctypes.c_int32(0), ctypes.c_int32(0)
    load().ctcb_last_walk_config(ctypes.byref(p), ctypes.byref(nw))
    return p.value, nw.value
