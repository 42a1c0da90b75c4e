"""CPU tests of the label-free decoding projection entry (ctcb_proj_greedy_decode, include/ctcb.h): the symbol is exported
and declared, the version is unchanged, and the entry refuses bad arguments -- NULL outputs or projection, an <unk> outside
the vocabulary, a bad operand type, misaligned K or strides, a T too long for the collapse kernel, host buffers -- with
the right status and message before it touches a device.  proj_greedy_decode has no CPU path."""
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


def test_greedy_entry_is_declared_and_exported(lib):
    with open(os.path.join(ROOT, "include", "ctcb.h")) as f:
        assert "int ctcb_proj_greedy_decode(" in f.read()
    assert "ctcb_proj_greedy_decode" in lib.EXPORTS and hasattr(lib.load(), "ctcb_proj_greedy_decode")
    assert lib.load().ctcb_version() == 103


def _args(lib, keep, T=140, V=46, K=64):
    """A decode problem on host arrays: every check before the device-memory ones passes."""
    B = 2
    h = np.zeros((B, T, K), np.float32)
    w = np.zeros((V, K), np.float32)
    toks = np.zeros((B, T), np.int32)
    lens = np.zeros((B,), np.int32)
    keep += [h, w, toks, lens]
    pj = lib.Proj()
    pj.hidden, pj.hidden_stride_t, pj.hidden_stride_b, pj.K = h.ctypes.data, K, T * K, K
    pj.weight = w.ctypes.data
    return pj, (T, B, V), toks.ctypes.data, lens.ctypes.data


def _call(l, pj, shape, unk, toks, lens, blank=0, lengths=None, ldt=0):
    T, B, V = shape
    return l.ctcb_proj_greedy_decode(ctypes.byref(pj) if pj is not None else None, T, B, V, lengths, ldt, blank, unk,
                                     toks, lens, None)


def _refused(l, lib, rc, status, text):
    assert rc == status, (rc, l.ctcb_last_error())
    assert text in l.ctcb_last_error(), l.ctcb_last_error()


def test_greedy_entry_refuses_bad_arguments_without_gpu(lib):
    l, keep = lib.load(), []
    pj, shape, t, n = _args(lib, keep)
    bad = lib.CTCB_INVALID_VALUE
    # NULL outputs and a NULL projection
    _refused(l, lib, _call(l, pj, shape, -1, None, n), bad, b"NULL")
    _refused(l, lib, _call(l, pj, shape, -1, t, None), bad, b"NULL")
    _refused(l, lib, _call(l, None, shape, -1, t, n), bad, b"NULL")
    # shapes
    for s in ((0, 2, 46), (140, 0, 46), (140, 2, 0)):
        _refused(l, lib, _call(l, pj, s, -1, t, n), bad, b"bad shape")
    # <unk> outside the vocabulary
    for unk in (shape[2], shape[2] + 7):
        _refused(l, lib, _call(l, pj, shape, unk, t, n), bad, b"unk")
    # a length dtype the parameter layer does not know (bf16 and beyond)
    _refused(l, lib, _call(l, pj, shape, -1, t, n, lengths=n, ldt=4), bad, b"length dtype")
    # the projection's own checks: operand type, 16-byte K and strides, NULL operands
    pj.operand_dtype = 2
    _refused(l, lib, _call(l, pj, shape, -1, t, n), bad, b"operand_dtype")
    pj.operand_dtype = 0
    for field, value in (("K", 62), ("hidden_stride_t", 66), ("hidden_stride_b", 140 * 64 + 2)):
        old = getattr(pj, field)
        setattr(pj, field, value)
        _refused(l, lib, _call(l, pj, shape, -1, t, n), bad, b"multiples of 16 bytes")
        setattr(pj, field, old)
    pj.operand_dtype = 1                 # bf16: K = 68 is 136 bytes, not a multiple of 16
    pj.K = 68
    _refused(l, lib, _call(l, pj, shape, -1, t, n), bad, b"multiples of 16 bytes")
    pj.operand_dtype, pj.K = 0, 64
    w = pj.weight
    pj.weight = None
    _refused(l, lib, _call(l, pj, shape, -1, t, n), bad, b"NULL")
    pj.weight = w
    # host buffers: there is no CPU path (every valid unk gets this far; -1 and below = no <unk> rule)
    for unk in (-5, -1, 0, 17, shape[2] - 1):
        _refused(l, lib, _call(l, pj, shape, unk, t, n), bad, b"device memory")
    # no V > 64 condition: V = 46 and V = 2 get as far as the buffers
    for V in (2, 46):
        _refused(l, lib, _call(l, pj, (shape[0], shape[1], V), -1, t, n), bad, b"device memory")


def test_greedy_entry_refuses_a_row_too_long_for_the_collapse_kernel(lib):
    l, keep = lib.load(), []
    pj, shape, t, n = _args(lib, keep, T=30000)
    _refused(l, lib, _call(l, pj, shape, -1, t, n), lib.CTCB_UNSUPPORTED, b"too long")


def test_proj_greedy_decode_refuses_cpu_tensors():
    torch = pytest.importorskip("torch")
    from gluon_e2e_asr_b200 import ProjCtcLoss, proj_greedy_decode
    h, w = torch.zeros((2, 10, 64)), torch.zeros((46, 64))
    with pytest.raises(RuntimeError) as e:
        proj_greedy_decode(h, w, None)
    assert "CPU" in str(e.value)
    with pytest.raises(RuntimeError) as e:
        ProjCtcLoss(64, 46).decode(h)
    assert "CPU" in str(e.value)
