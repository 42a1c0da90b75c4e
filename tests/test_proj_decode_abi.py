"""CPU tests of the decoding projection entry (ctcb_proj_forward_decode, include/ctcb.h): the symbol is exported and
declared, and the entry refuses bad decode arguments -- NULL outputs, an <unk> outside the vocabulary, a T too long for
the collapse kernel, host outputs -- before it touches a device.  proj_ctc_eval has no CPU path."""
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


def test_decode_entry_is_declared_and_exported(lib):
    with open(os.path.join(ROOT, "include", "ctcb.h")) as f:
        assert "int ctcb_proj_forward_decode(" in f.read()
    assert "ctcb_proj_forward_decode" in lib.EXPORTS and hasattr(lib.load(), "ctcb_proj_forward_decode")
    assert lib.load().ctcb_version() == 103


def _args(lib, keep, T=140, V=300):
    """A projection problem on host arrays: every check before the decode's own ones would pass on shape."""
    B, K, L = 2, 64, 4
    h = np.zeros((B, T, K), np.float32)
    w = np.zeros((V, K), np.float32)
    lab = np.ones((B, L), np.int32)
    loss = np.zeros((B,), np.float32)
    toks = np.zeros((B, T), np.int32)
    lens = np.zeros((B,), np.int32)
    keep += [h, w, lab, loss, toks, lens]
    pj = lib.Proj()
    pj.hidden, pj.hidden_stride_t, pj.hidden_stride_b, pj.K = h.ctypes.data, K, T * K, K
    pj.weight = w.ctypes.data
    p = lib.Problem()
    p.T, p.B, p.V, p.Lmax, p.blank = T, B, V, L, 0
    p.labels, p.label_dtype, p.label_stride_b, p.label_stride_l = lab.ctypes.data, lib.DT_I32, L, 1
    p.loss = loss.ctypes.data
    return pj, p, toks, lens


def _call(l, pj, p, unk, toks, lens):
    return l.ctcb_proj_forward_decode(ctypes.byref(pj) if pj is not None else None, ctypes.byref(p), 0, unk,
                                      toks, lens, None, 0, None)


def test_decode_entry_refuses_bad_arguments_without_gpu(lib):
    l, keep = lib.load(), []
    pj, p, toks, lens = _args(lib, keep)
    t, n = toks.ctypes.data, lens.ctypes.data
    # NULL outputs
    assert _call(l, pj, p, -1, None, n) == lib.CTCB_INVALID_VALUE
    assert b"NULL" in l.ctcb_last_error()
    assert _call(l, pj, p, -1, t, None) == lib.CTCB_INVALID_VALUE
    # <unk> outside the vocabulary
    for unk in (p.V, p.V + 7):
        assert _call(l, pj, p, unk, t, n) == lib.CTCB_INVALID_VALUE
        assert b"unk" in l.ctcb_last_error()
    # host outputs: there is no CPU path (every valid unk gets this far, -1 and below = no <unk> rule)
    for unk in (-5, -1, 0, 17, p.V - 1):
        assert _call(l, pj, p, unk, t, n) == lib.CTCB_INVALID_VALUE
        assert b"device memory" in l.ctcb_last_error()
    # a NULL projection or problem: ctcb_proj_forward's own checks
    assert _call(l, None, p, -1, t, n) == lib.CTCB_INVALID_VALUE


def test_decode_entry_refuses_a_row_too_long_for_the_collapse_kernel(lib):
    l, keep = lib.load(), []
    pj, p, toks, lens = _args(lib, keep, T=30000)
    assert _call(l, pj, p, -1, toks.ctypes.data, lens.ctypes.data) == lib.CTCB_UNSUPPORTED
    assert b"too long" in l.ctcb_last_error()


def test_proj_ctc_eval_refuses_cpu_tensors():
    torch = pytest.importorskip("torch")
    from gluon_e2e_asr_b200 import proj_ctc_eval
    h, w = torch.zeros((2, 10, 64)), torch.zeros((300, 64))
    lab = torch.ones((2, 3), dtype=torch.int32)
    with pytest.raises(RuntimeError) as e:
        proj_ctc_eval(h, w, None, lab)
    assert "CPU" in str(e.value)
