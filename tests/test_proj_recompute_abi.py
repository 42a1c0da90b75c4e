"""CPU tests of the recomputing backward of the fused projection (ctcb_proj_backward, include/ctcb.h): the symbol is
declared, exported and bound, the library version is unchanged, and the entry refuses bad arguments -- NULLs, bad shapes,
vocabularies the fused projection does not take, a missing / small / misaligned workspace, host memory -- before it
touches a device.  The training call keeps using ctcb_workspace_bytes(need_grad=1): no new size query."""
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


def test_backward_entry_is_declared_exported_and_bound(lib):
    with open(os.path.join(ROOT, "include", "ctcb.h")) as f:
        assert "int ctcb_proj_backward(" in f.read()
    l = lib.load()
    assert "ctcb_proj_backward" in lib.EXPORTS and hasattr(l, "ctcb_proj_backward")
    assert l.ctcb_proj_backward.argtypes is not None and len(l.ctcb_proj_backward.argtypes) == 5
    assert l.ctcb_version() == 103


def _args(lib, keep, T=140, V=300, L=4, K=64):
    """A projection problem on host arrays, with a gradient buffer: every shape check would pass."""
    B = 2
    h = np.zeros((B, T, K), np.float32)
    w = np.zeros((V, K), np.float32)
    lab = np.ones((B, L), np.int32)
    loss = np.zeros((B,), np.float32)
    grad = np.zeros((B, T, V), np.float32)
    keep += [h, w, lab, loss, grad]
    pj = lib.Proj()
    pj.hidden, pj.hidden_stride_t, pj.hidden_stride_b, pj.K = h.ctypes.data, K, T * K, K
    pj.weight = w.ctypes.data
    p = lib.Problem()
    p.T, p.B, p.V, p.Lmax, p.blank = T, B, V, L, 0
    p.labels, p.label_dtype, p.label_stride_b, p.label_stride_l = lab.ctypes.data, lib.DT_I32, L, 1
    p.loss = loss.ctypes.data
    p.grad, p.grad_stride_t, p.grad_stride_b = grad.ctypes.data, V, T * V
    return pj, p


def _call(l, pj, p, ws=None, nbytes=0):
    return l.ctcb_proj_backward(ctypes.byref(pj) if pj is not None else None, ctypes.byref(p) if p is not None else None,
                                ws, nbytes, None)


def test_backward_entry_refuses_bad_arguments_without_gpu(lib):
    l, keep = lib.load(), []
    pj, p = _args(lib, keep)
    need = lib.workspace_bytes(p.T, p.B, p.V, p.Lmax, True)
    # NULL projection / problem
    assert _call(l, None, p) == lib.CTCB_INVALID_VALUE
    assert _call(l, pj, None) == lib.CTCB_INVALID_VALUE
    # NULL gradient buffer
    p.grad = None
    assert _call(l, pj, p) == lib.CTCB_INVALID_VALUE
    assert b"grad" in l.ctcb_last_error()
    pj, p = _args(lib, keep)
    # bad shapes and a blank outside the vocabulary (validate, as every entry)
    for field, value in (("T", 0), ("B", 0), ("V", 1), ("Lmax", -1), ("blank", 300)):
        pj, p = _args(lib, keep)
        setattr(p, field, value)
        assert _call(l, pj, p) == lib.CTCB_INVALID_VALUE, field
    # NULL labels with a label row
    pj, p = _args(lib, keep)
    p.labels = None
    assert _call(l, pj, p) == lib.CTCB_INVALID_VALUE
    # workspace: NULL, too small, misaligned (checked before any device pointer)
    pj, p = _args(lib, keep)
    assert _call(l, pj, p, None, need) == lib.CTCB_INVALID_VALUE
    assert b"workspace" in l.ctcb_last_error()
    ws = np.zeros(need + 512, np.uint8)
    keep.append(ws)
    base = (ws.ctypes.data + 255) // 256 * 256
    assert _call(l, pj, p, base, need - 1) == lib.CTCB_WORKSPACE_TOO_SMALL
    assert _call(l, pj, p, base + 8, need) == lib.CTCB_INVALID_VALUE
    assert b"aligned" in l.ctcb_last_error()
    # host memory: there is no CPU path
    assert _call(l, pj, p, base, need) == lib.CTCB_INVALID_VALUE
    assert b"device memory" in l.ctcb_last_error()


@pytest.mark.parametrize("V, L", [(46, 4), (64, 4), (120, 119), (100, 150)])
def test_backward_entry_is_unsupported_where_the_forward_is(lib, V, L):
    """V <= 64 or V <= Lmax + 1: the fused projection is not used there, and neither is its backward."""
    l, keep = lib.load(), []
    pj, p = _args(lib, keep, V=V, L=L)
    assert _call(l, pj, p) == lib.CTCB_UNSUPPORTED
    assert b"V > 64" in l.ctcb_last_error()


def test_recompute_forward_refuses_what_its_backward_cannot_take(lib):
    """proj_ctas=1: the backward's kernel does not fit shared memory once Lp + NT > 2020 (label-row words, 256-column
    vocabulary tiles); at Lmax = 4 that is V > 256 * 2016.  ctcb_proj_forward(keep_for_backward=1, logits NULL) refuses such
    a shape before it looks at the workspace, with the backward's error; one vocabulary tile fewer, without
    keep_for_backward, or with CTA pairs, the shape passes that check (and these host buffers fail at the workspace)."""
    l, keep = lib.load(), []
    pj, p = _args(lib, keep)                     # host buffers of a small shape: only the shape fields change below
    p.grad = None

    def forward(V, keep_for_backward):
        p.V = V
        return l.ctcb_proj_forward(ctypes.byref(pj), ctypes.byref(p), keep_for_backward, None, 0, None)

    limit = 256 * (2020 - 4)
    with lib.options(proj_ctas=1):
        assert forward(limit + 1, 1) == lib.CTCB_UNSUPPORTED
        assert b"shared memory" in l.ctcb_last_error()
        for V, k in ((limit, 1), (limit + 1, 0)):
            assert forward(V, k) == lib.CTCB_INVALID_VALUE and b"workspace" in l.ctcb_last_error(), (V, k)
    with lib.options(proj_ctas=2):
        assert forward(limit + 1, 1) == lib.CTCB_INVALID_VALUE and b"workspace" in l.ctcb_last_error()


def test_recompute_option_is_validated_and_has_no_cpu_path():
    torch = pytest.importorskip("torch")
    from gluon_e2e_asr_b200 import proj_ctc_loss
    h, w = torch.zeros((2, 10, 64), requires_grad=True), torch.zeros((300, 64))
    lab = torch.ones((2, 3), dtype=torch.int32)
    with pytest.raises(ValueError):
        proj_ctc_loss(h, w, None, lab, fused_training="recompte")
    with pytest.raises(RuntimeError) as e:
        proj_ctc_loss(h, w, None, lab, fused_training="recompute")
    assert "CPU" in str(e.value)
