"""CPU tests of the decoding loss evaluation (ctcb_forward_decode_typed, include/ctcb.h): the symbol is exported and
declared, and the entry refuses bad arguments -- NULL outputs, a bad problem, an <unk> outside the vocabulary, a T too
long for the collapse kernel, a logits dtype other than fp32 / bf16, host buffers -- before it touches a device.
ctc_eval and CtcLoss.evaluate have no CPU path."""
import ctypes
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build_cuda()
    from gluon_e2e_asr_b200 import _lib
    return _lib


def test_entry_is_declared_and_exported(lib):
    with open(os.path.join(ROOT, "include", "ctcb.h")) as f:
        assert "int ctcb_forward_decode_typed(" in f.read()
    assert "ctcb_forward_decode_typed" in lib.EXPORTS and hasattr(lib.load(), "ctcb_forward_decode_typed")
    assert lib.load().ctcb_version() == 103


def _args(lib, keep, T=50, V=46):
    """A loss problem on host arrays: every check before the decode's own ones would pass on shape."""
    B, L = 2, 4
    x = np.zeros((B, T, V), np.float32)
    lab = np.ones((B, L), np.int32)
    loss = np.zeros((B,), np.float32)
    toks = np.zeros((B, T), np.int32)
    lens = np.zeros((B,), np.int32)
    keep += [x, lab, loss, toks, lens]
    p = lib.Problem()
    p.T, p.B, p.V, p.Lmax, p.blank = T, B, V, L, 0
    p.logits, p.logits_stride_t, p.logits_stride_b = x.ctypes.data, V, T * V
    p.labels, p.label_dtype, p.label_stride_b, p.label_stride_l = lab.ctypes.data, lib.DT_I32, L, 1
    p.loss = loss.ctypes.data
    return p, toks.ctypes.data, lens.ctypes.data


def _call(l, p, unk, toks, lens, dtype=None, lib=None):
    return l.ctcb_forward_decode_typed(ctypes.byref(p) if p is not None else None, lib.DT_F32 if dtype is None else dtype,
                                       unk, toks, lens, None, 0, None)


def test_entry_refuses_bad_arguments_without_gpu(lib):
    l, keep = lib.load(), []
    p, t, n = _args(lib, keep)
    call = lambda p_, unk, t_, n_, dtype=None: _call(l, p_, unk, t_, n_, dtype, lib)
    # NULL outputs
    assert call(p, -1, None, n) == lib.CTCB_INVALID_VALUE
    assert b"NULL" in l.ctcb_last_error()
    assert call(p, -1, t, None) == lib.CTCB_INVALID_VALUE
    # the problem checks of ctcb_forward_typed
    assert call(None, -1, t, n) == lib.CTCB_INVALID_VALUE
    assert b"problem is NULL" in l.ctcb_last_error()
    bad = lib.Problem.from_buffer_copy(p)
    bad.blank = p.V
    assert call(bad, -1, t, n) == lib.CTCB_INVALID_VALUE
    assert b"blank" in l.ctcb_last_error()
    # <unk> outside the vocabulary
    for unk in (p.V, p.V + 7):
        assert call(p, unk, t, n) == lib.CTCB_INVALID_VALUE
        assert b"unk" in l.ctcb_last_error()
    # a logits dtype other than fp32 / bf16 (fp16 is not supported)
    for dtype in (lib.DT_I32, lib.DT_F64, 5, -1):
        assert call(p, -1, t, n, dtype) == lib.CTCB_INVALID_VALUE
        assert b"neither CTCB_F32 nor CTCB_BF16" in l.ctcb_last_error()
    # host buffers: there is no CPU path (every valid unk and both logits dtypes get this far)
    for unk in (-5, -1, 0, 17, p.V - 1):
        for dtype in (lib.DT_F32, lib.DT_BF16):
            assert call(p, unk, t, n, dtype) == lib.CTCB_INVALID_VALUE
            assert b"device memory" in l.ctcb_last_error()


def test_entry_refuses_a_row_too_long_for_the_collapse_kernel(lib):
    l, keep = lib.load(), []
    p, t, n = _args(lib, keep, T=30000, V=4)
    assert _call(l, p, -1, t, n, lib=lib) == lib.CTCB_UNSUPPORTED
    assert b"too long" in l.ctcb_last_error()


def test_ctc_eval_refuses_cpu_tensors():
    torch = pytest.importorskip("torch")
    from gluon_e2e_asr_b200 import CtcLoss, ctc_eval
    x = torch.zeros((2, 10, 46))
    lab = torch.ones((2, 3), dtype=torch.int32)
    with pytest.raises(RuntimeError) as e:
        ctc_eval(x, lab)
    assert "CPU" in str(e.value)
    with pytest.raises(RuntimeError):
        CtcLoss().evaluate(x, lab)
