"""CPU tests of the bfloat16 logits entries (include/ctcb.h, *_typed): the binding's constant and symbol list match the
header, and the typed entries refuse bad arguments -- an unknown logits type, bf16 labels or lengths, a NULL problem --
with CTCB_INVALID_VALUE before they touch a device."""
import ctypes
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build_cuda()
    from gluon_e2e_asr_b200 import _lib
    return _lib


def test_bf16_constant_matches_header(lib):
    with open(os.path.join(ROOT, "include", "ctcb.h")) as f:
        src = f.read()
    m = re.search(r"\bCTCB_BF16\s*=\s*(\d+)", src)
    assert m and int(m.group(1)) == lib.DT_BF16
    for name in ("ctcb_loss_grad_typed", "ctcb_forward_typed", "ctcb_backward_typed", "ctcb_greedy_decode_typed"):
        assert name in lib.EXPORTS and hasattr(lib.load(), name)


def _valid_problem(lib, keep):
    """A problem that passes every check up to the logits type (host arrays: nothing reaches a device)."""
    x = np.zeros((2, 3, 4), np.float32)
    lab = np.zeros((2, 2), np.int32)
    loss = np.zeros((2,), np.float32)
    keep += [x, lab, loss]
    p = lib.Problem()
    p.T, p.B, p.V, p.Lmax, p.blank = 3, 2, 4, 2, 0
    p.logits, p.logits_stride_t, p.logits_stride_b = x.ctypes.data, 4, 12
    p.labels, p.label_dtype, p.label_stride_b, p.label_stride_l = lab.ctypes.data, lib.DT_I32, 2, 1
    p.loss = loss.ctypes.data
    return p


def _typed_calls(l, p):
    ref = ctypes.byref(p) if p is not None else None
    return {
        "loss_grad": lambda dt: l.ctcb_loss_grad_typed(ref, dt, None, 0, None),
        "forward": lambda dt: l.ctcb_forward_typed(ref, dt, 1, None, 0, None),
        "backward": lambda dt: l.ctcb_backward_typed(ref, dt, None, 0, None),
    }


def test_typed_entries_refuse_an_unknown_logits_dtype(lib):
    l, keep = lib.load(), []
    p = _valid_problem(lib, keep)
    for name, call in _typed_calls(l, p).items():
        for dt in (-1, lib.DT_I32, lib.DT_I64, lib.DT_F64, 5, 99):
            assert call(dt) == lib.CTCB_INVALID_VALUE, (name, dt)
            assert b"logits dtype" in l.ctcb_last_error(), (name, dt)
    # the valid types get past the type check and stop at the (missing) workspace
    for dt in (lib.DT_F32, lib.DT_BF16):
        assert l.ctcb_loss_grad_typed(ctypes.byref(p), dt, None, 0, None) == lib.CTCB_INVALID_VALUE
        assert b"workspace" in l.ctcb_last_error()


def test_typed_entries_refuse_bf16_labels_and_lengths(lib):
    l, keep = lib.load(), []
    for field in ("label_dtype", "data_lengths_dtype", "label_lengths_dtype"):
        p = _valid_problem(lib, keep)
        n = np.zeros((2,), np.int32)
        keep.append(n)
        p.data_lengths, p.label_lengths = n.ctypes.data, n.ctypes.data
        p.data_lengths_dtype = p.label_lengths_dtype = lib.DT_I32
        setattr(p, field, lib.DT_BF16)
        for name, call in _typed_calls(l, p).items():
            assert call(lib.DT_BF16) == lib.CTCB_INVALID_VALUE, (field, name)
            assert b"label/length dtype" in l.ctcb_last_error(), (field, name)
        assert l.ctcb_loss_grad(ctypes.byref(p), None, 0, None) == lib.CTCB_INVALID_VALUE


def test_typed_entries_refuse_a_null_problem(lib):
    l = lib.load()
    for name, call in _typed_calls(l, None).items():
        assert call(lib.DT_BF16) == lib.CTCB_INVALID_VALUE, name
        assert b"NULL" in l.ctcb_last_error(), name


def test_typed_decode_refuses_bad_arguments(lib):
    l = lib.load()
    x = np.zeros((2, 3, 4), np.float32)
    toks = np.zeros((2, 3), np.int32)
    lens = np.zeros((2,), np.int32)
    args = lambda dt: l.ctcb_greedy_decode_typed(x.ctypes.data, dt, 4, 12, None, 0, 3, 2, 4, 0, -1,
                                                 toks.ctypes.data, lens.ctypes.data, None)
    for dt in (lib.DT_I32, lib.DT_F64, 5):
        assert args(dt) == lib.CTCB_INVALID_VALUE
        assert b"logits dtype" in l.ctcb_last_error()
    # valid types: refused for host memory (there is no CPU path), not for their type
    for dt in (lib.DT_F32, lib.DT_BF16):
        assert args(dt) == lib.CTCB_INVALID_VALUE
        assert b"device memory" in l.ctcb_last_error()
    assert l.ctcb_greedy_decode_typed(None, lib.DT_BF16, 4, 12, None, 0, 3, 2, 4, 0, -1, toks.ctypes.data,
                                      lens.ctypes.data, None) == lib.CTCB_INVALID_VALUE


def test_python_layer_names_fp16_in_its_refusal():
    torch = pytest.importorskip("torch")
    from gluon_e2e_asr_b200 import ops
    x = torch.zeros((2, 3, 4), dtype=torch.float16)
    with pytest.raises((TypeError, RuntimeError)) as e:
        ops._check_data(x)
    # without a GPU the CPU tensor is refused first; the dtype message is checked on the GPU (tests/test_bf16_gpu.py)
    assert "CUDA" in str(e.value) or "float16" in str(e.value)
