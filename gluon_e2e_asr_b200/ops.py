"""The raw operator surface of the reference's CTC path on torch CUDA tensors.

``ctc_loss`` mirrors ``mx.nd.contrib.ctc_loss`` exactly as the reference calls it at
/root/reference/scripts/swbd/loss.py:134-139 (same argument names, meaning and defaults;
alias ``CTCLoss`` like upstream).  torch is only plumbing here: device memory, the current
stream and autograd bookkeeping.  All arithmetic happens in libctcb.so's sm_100a kernels,
reached through ctypes with either DLPack structs (default, ``handoff='dlpack'``) or raw
pointers (``handoff='pointer'``); without the built library or without a CUDA tensor the
call raises -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes
import os

import torch
from torch.utils import dlpack as _dlpack

from . import _lib

__all__ = ["ctc_loss", "CTCLoss", "ctc_loss_and_grad", "ctc_eval", "greedy_decode", "workspace_bytes"]

_DT = {torch.int32: _lib.DT_I32, torch.int64: _lib.DT_I64, torch.float32: _lib.DT_F32, torch.float64: _lib.DT_F64}
# logits element types: float32, and bfloat16 (a mixed-precision model's logits; loss fp32, gradient bf16 -- include/ctcb.h)
_DT_LOGITS = {torch.float32: _lib.DT_F32, torch.bfloat16: _lib.DT_BF16}
_HANDOFF = os.environ.get("CTCB_HANDOFF", "dlpack")

_PyCapsule_GetPointer = ctypes.pythonapi.PyCapsule_GetPointer
_PyCapsule_GetPointer.restype = ctypes.c_void_p
_PyCapsule_GetPointer.argtypes = [ctypes.py_object, ctypes.c_char_p]


def workspace_bytes(T, B, V, Lmax, need_grad=True):
    return _lib.workspace_bytes(T, B, V, Lmax, need_grad)


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_cur_device = getattr(torch._C, "_cuda_getDevice", None)


def _stream_ptr(device):
    """cudaStream_t of torch's current stream on ``device`` (host-side plumbing, kept cheap)."""
    if _raw_stream is not None:
        return _raw_stream(device.index)
    return torch.cuda.current_stream(device).cuda_stream


class _on_device:
    """``with torch.cuda.device(d)`` only when ``d`` is not already current."""
    __slots__ = ("ctx",)

    def __init__(self, device):
        same = _cur_device is not None and _cur_device() == device.index
        self.ctx = None if same else torch.cuda.device(device)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
        return False


def _as_index_tensor(x, device, name):
    """labels / lengths: any float or int dtype (the reference delivers float32,
    reader_kaldi_io.py:33-35, batchify.py:78-82); other dtypes are cast to float32/int64."""
    if x is None:
        return None
    if not isinstance(x, torch.Tensor):
        x = torch.as_tensor(x)
    if x.device != device:
        raise ValueError("%s is on %s but data is on %s" % (name, x.device, device))
    if x.dtype not in _DT:
        x = x.to(torch.float32 if x.dtype.is_floating_point else torch.int64)
    return x


def _check_data(data):
    if not isinstance(data, torch.Tensor):
        raise TypeError("data must be a torch.Tensor")
    if not data.is_cuda:
        raise RuntimeError("gluon_e2e_asr_b200.ctc_loss has no CPU path: data must be a CUDA tensor")
    if data.dim() != 3:
        raise ValueError("data must be 3-d, got shape %s" % (tuple(data.shape),))
    if data.dtype not in _DT_LOGITS:
        raise TypeError("data must be float32 (the reference's logits dtype) or bfloat16, got %s "
                        "(float16 logits are not supported: cast them to bfloat16 or float32)" % data.dtype)
    if data.shape[2] > 1 and data.stride(2) != 1:
        data = data.contiguous()
    return data


class _Call:
    """One operator call, prepared once and handed to the library through either hand-off."""

    def __init__(self, data, label, data_lengths, label_lengths, blank_last, ntc, tn):
        self.data = data
        self.ldt = _DT_LOGITS[data.dtype]          # element type of the logits and of the gradient
        self.ntc, self.tn, self.blank_last = ntc, tn, blank_last
        dev = data.device
        self.label = _as_index_tensor(label, dev, "label")
        if self.label.dim() != 2:
            raise ValueError("label must be 2-d")
        self.data_lengths = _as_index_tensor(data_lengths, dev, "data_lengths")
        self.label_lengths = _as_index_tensor(label_lengths, dev, "label_lengths")
        ta, ba = (1, 0) if ntc else (0, 1)
        self.T, self.B, self.V = data.shape[ta], data.shape[ba], data.shape[2]
        lb, ll = (1, 0) if tn else (0, 1)
        if self.label.shape[lb] != self.B:
            raise ValueError("label batch %d != data batch %d" % (self.label.shape[lb], self.B))
        self.Lmax = self.label.shape[ll]
        for n, v in (("data_lengths", self.data_lengths), ("label_lengths", self.label_lengths)):
            if v is not None:
                if v.dim() != 1 or v.shape[0] != self.B:
                    raise ValueError("%s must have shape (%d,)" % (n, self.B))
        if self.data_lengths is not None:
            self.data_lengths = self.data_lengths.contiguous()
        if self.label_lengths is not None:
            self.label_lengths = self.label_lengths.contiguous()
        self._axes = (ta, ba, lb, ll)

    def flags(self):
        return (_lib.LAYOUT_NTC if self.ntc else 0) | (_lib.LABEL_TN if self.tn else 0)

    def problem(self, loss, grad=None, head=None, loss_sum=None, status=None):
        ta, ba, lb, ll = self._axes
        p = _lib.Problem()
        p.T, p.B, p.V, p.Lmax = self.T, self.B, self.V, self.Lmax
        p.blank = self.V - 1 if self.blank_last else 0
        p.label_pad = -1 if self.blank_last else 0
        d = self.data
        p.logits, p.logits_stride_t, p.logits_stride_b = d.data_ptr(), d.stride(ta), d.stride(ba)
        if grad is not None:
            p.grad, p.grad_stride_t, p.grad_stride_b = grad.data_ptr(), grad.stride(ta), grad.stride(ba)
        lab = self.label
        p.labels, p.label_dtype = lab.data_ptr(), _DT[lab.dtype]
        p.label_stride_b, p.label_stride_l = lab.stride(lb), lab.stride(ll)
        if self.data_lengths is not None:
            p.data_lengths, p.data_lengths_dtype = self.data_lengths.data_ptr(), _DT[self.data_lengths.dtype]
        if self.label_lengths is not None:
            p.label_lengths, p.label_lengths_dtype = self.label_lengths.data_ptr(), _DT[self.label_lengths.dtype]
        if head is not None:
            p.head_grad = head.data_ptr()
        p.loss = loss.data_ptr()
        if loss_sum is not None:
            p.loss_sum = loss_sum.data_ptr()
        if status is not None:
            p.status = status.data_ptr()
        return p

    def run(self, phase, ws, loss, grad=None, head=None, loss_sum=None, status=None, keep=False, handoff=None):
        lib = _lib.load()
        stream = _stream_ptr(self.data.device)
        handoff = handoff or _HANDOFF
        with _on_device(self.data.device):
            if handoff == "dlpack" and status is None:
                caps = []

                def cap(t):
                    if t is None:
                        return None
                    c = _dlpack.to_dlpack(t)
                    caps.append(c)               # keeps the DLManagedTensor alive for the call
                    return _PyCapsule_GetPointer(c, b"dltensor")
                flags = self.flags() | phase | (_lib.KEEP_FOR_BACKWARD if keep else 0)
                rc = lib.ctcb_loss_grad_dlpack(cap(self.data), cap(self.label), cap(self.data_lengths),
                                               cap(self.label_lengths), cap(head), cap(loss), cap(grad),
                                               cap(loss_sum), 1 if self.blank_last else 0, flags,
                                               ws.data_ptr(), ws.numel(), stream)
                del caps
            else:
                p = self.problem(loss, grad, head, loss_sum, status)
                if phase == _lib.PHASE_FORWARD:
                    rc = lib.ctcb_forward_typed(ctypes.byref(p), self.ldt, 1 if keep else 0, ws.data_ptr(), ws.numel(), stream)
                elif phase == _lib.PHASE_BACKWARD:
                    rc = lib.ctcb_backward_typed(ctypes.byref(p), self.ldt, ws.data_ptr(), ws.numel(), stream)
                else:
                    rc = lib.ctcb_loss_grad_typed(ctypes.byref(p), self.ldt, ws.data_ptr(), ws.numel(), stream)
        _lib.check(rc)


def _alloc_ws(call, need_grad):
    n = _lib.workspace_bytes(call.T, call.B, call.V, call.Lmax, need_grad)
    return torch.empty((n,), dtype=torch.uint8, device=call.data.device)


# Forward of a differentiable call: small problems run the fused forward+gradient once (the
# gradient is stored like MXNet's operator stores it, SURVEY 8a row a8) and Backward only scales
# it by the head gradient; large ones keep the alpha/beta history and write head*G once in
# Backward, which saves a pass over the (T,B,V) gradient.  bfloat16 logits always take the second
# branch: scaling a stored bf16 gradient would round every element twice.
_FUSE_IN_FORWARD_MAX_ELEMS = 8 * 1024 * 1024


class _CtcLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, data, label, data_lengths, label_lengths, blank_last, ntc, tn):
        call = _Call(data, label, data_lengths, label_lengths, blank_last, ntc, tn)
        need = ctx.needs_input_grad[0]
        loss = torch.empty((call.B,), dtype=torch.float32, device=data.device)
        ctx.call = call
        if need and data.dtype == torch.float32 and data.numel() <= _FUSE_IN_FORWARD_MAX_ELEMS:
            grad = torch.empty_like(data)           # same layout as the logits: no swapaxes backward
            call.run(_lib.PHASE_FUSED, _cached_ws(call, data.device), loss, grad=grad)
            ctx.grad, ctx.ws = grad, None
        else:
            ws = _alloc_ws(call, need)              # holds the history until backward: not shared
            call.run(_lib.PHASE_FORWARD, ws, loss, keep=need)
            ctx.grad, ctx.ws = None, ws
        return loss

    @staticmethod
    def backward(ctx, head):
        call = ctx.call
        if head.dtype != torch.float32 or not head.is_contiguous():
            head = head.to(torch.float32).contiguous()
        if ctx.grad is not None:
            grad, ctx.grad = ctx.grad, None
            ta, ba = call._axes[0], call._axes[1]
            with _on_device(grad.device):
                _lib.check(_lib.load().ctcb_scale_rows(grad.data_ptr(), grad.stride(ta), grad.stride(ba), call.T, call.B,
                                                       call.V, head.data_ptr(), _stream_ptr(grad.device)))
            return grad, None, None, None, None, None, None
        ws = ctx.ws
        if ws is None:
            raise RuntimeError("ctc_loss: backward called twice (the workspace is released after the first)")
        grad = torch.empty_like(call.data)
        loss_scratch = torch.empty((call.B,), dtype=torch.float32, device=head.device)
        call.run(_lib.PHASE_BACKWARD, ws, loss_scratch, grad=grad, head=head)
        ctx.ws = None
        return grad, None, None, None, None, None, None


def _blank_last(blank_label):
    if blank_label not in ("first", "last"):
        raise ValueError("blank_label must be 'first' or 'last', got %r" % (blank_label,))
    return blank_label == "last"


def ctc_loss(data, label, data_lengths=None, label_lengths=None, use_data_lengths=False,
             use_label_lengths=False, blank_label="first"):
    """``mx.nd.contrib.ctc_loss`` as called at scripts/swbd/loss.py:134-139.

    data (T, B, V) float32 or bfloat16 CUDA logits (softmax is inside; bf16: fp32 loss, bf16 gradient);
    label (B, Lmax) any numeric dtype,
    truncated to int; lengths (B,) used only when the matching ``use_*`` flag is set
    (otherwise T, resp. the first padding value: 0 for blank_label='first', -1 for 'last').
    Returns the per-utterance negative log-likelihood (B,); differentiable w.r.t. ``data``.
    """
    data = _check_data(data)
    if use_data_lengths and data_lengths is None:
        raise ValueError("use_data_lengths=True needs data_lengths")
    if use_label_lengths and label_lengths is None:
        raise ValueError("use_label_lengths=True needs label_lengths")
    return _CtcLossFn.apply(data, label, data_lengths if use_data_lengths else None,
                            label_lengths if use_label_lengths else None,
                            _blank_last(blank_label), False, False)


CTCLoss = ctc_loss   # upstream alias: mx.nd.contrib.CTCLoss


def _ctc_loss_layout(pred, label, pred_lengths, label_lengths, blank_label, layout, label_layout):
    pred = _check_data(pred)
    return _CtcLossFn.apply(pred, label, pred_lengths, label_lengths, _blank_last(blank_label),
                            layout == "NTC", label_layout == "TN")


_ws_cache = {}


def _cached_ws(call, dev):
    """Scratch workspace per (device, stream, shape): calls on one stream are ordered, so the fused
    forward+gradient may reuse it from call to call."""
    key = (dev.index, _stream_ptr(dev), call.T, call.B, call.V, call.Lmax)
    ws = _ws_cache.get(key)
    if ws is None:
        ws = _ws_cache[key] = _alloc_ws(call, True)
    return ws


def ctc_loss_and_grad(pred, label, pred_lengths=None, label_lengths=None, head_grad=None,
                      blank_label="first", layout="NTC", label_layout="NT", loss_sum=None,
                      status=None, out_loss=None, out_grad=None, handoff=None):
    """Fused forward+backward (one ``ctcb_loss_grad`` call): returns (loss (B,), grad like pred).

    ``head_grad`` (B,) is the upstream gradient of each loss (``1/B`` for the reference's
    ``.mean().backward()``, train_ctc_ce.py:363-366); ``loss_sum`` an optional float64 device
    scalar accumulated in place.  The workspace is cached per (device, stream, shape).  bfloat16
    ``pred``: the loss is float32 and the gradient bfloat16 (``out_grad`` must then be bfloat16).
    """
    pred = _check_data(pred)
    if out_grad is not None and out_grad.dtype != pred.dtype:
        raise TypeError("out_grad must have the logits' dtype %s, got %s" % (pred.dtype, out_grad.dtype))
    call = _Call(pred, label, pred_lengths, label_lengths, _blank_last(blank_label),
                 layout == "NTC", label_layout == "TN")
    dev = pred.device
    ws = _cached_ws(call, dev)
    loss = out_loss if out_loss is not None else torch.empty((call.B,), dtype=torch.float32, device=dev)
    grad = out_grad if out_grad is not None else torch.empty_like(pred)
    if head_grad is not None:
        head_grad = head_grad.to(torch.float32).contiguous()
    call.run(_lib.PHASE_FUSED, ws, loss, grad=grad, head=head_grad, loss_sum=loss_sum, status=status,
             handoff=handoff)
    return loss, grad


def ctc_eval(pred, label, pred_lengths=None, label_lengths=None, blank_label="first", layout="NTC",
             label_layout="NT", unk=None):
    """The validation pass over logits (train_ctc_ce.py:143-160) in one read of them: ``(loss (B,), tokens (B,T) int32,
    lengths (B,) int32)``.

    ``loss`` is bit-identical to the loss ``ctc_loss`` computes under ``torch.no_grad()``; ``tokens`` / ``lengths`` are
    bit-identical to ``greedy_decode(pred, pred_lengths, blank, layout, unk)`` (blank 0, or V - 1 for
    ``blank_label="last"``).  The kernel pass that reads each logits row for the loss also keeps its best two symbols, and
    a small kernel collapses repeats and blanks (``ctcb_forward_decode_typed``).  float32 or bfloat16 ``pred``; no autograd
    graph.  The outputs go straight into ``edit_distance``."""
    pred = _check_data(pred)
    call = _Call(pred, label, pred_lengths, label_lengths, _blank_last(blank_label), layout == "NTC", label_layout == "TN")
    dev = pred.device
    ws = _alloc_ws(call, False)                 # the loss evaluation's size: no history
    loss = torch.empty((call.B,), dtype=torch.float32, device=dev)
    tokens = torch.empty((call.B, call.T), dtype=torch.int32, device=dev)
    lengths = torch.empty((call.B,), dtype=torch.int32, device=dev)
    p = call.problem(loss)
    with _on_device(dev):
        rc = _lib.load().ctcb_forward_decode_typed(ctypes.byref(p), call.ldt, -1 if unk is None else int(unk),
                                                   tokens.data_ptr(), lengths.data_ptr(), ws.data_ptr(), ws.numel(),
                                                   _stream_ptr(dev))
    _lib.check(rc)
    return loss, tokens, lengths


def greedy_decode(pred, pred_lengths=None, blank=0, layout="NTC", unk=None):
    """Greedy CTC decode of train_ctc_ce.py:149-160: argmax over V, collapse repeats, drop
    blank.  ``unk`` (the index of ``<unk>``): decode_ctc.py:120-140's rule -- a frame whose best symbol
    is ``unk`` takes its second best; the repeat test still compares with the raw best symbol of the
    previous frame.  ``pred`` float32 or bfloat16.  Returns (tokens (B,T) int32 -- prefix valid, lengths (B,) int32) on
    pred's device."""
    pred = _check_data(pred)
    ta, ba = (1, 0) if layout == "NTC" else (0, 1)
    T, B, V = pred.shape[ta], pred.shape[ba], pred.shape[2]
    pl = _as_index_tensor(pred_lengths, pred.device, "pred_lengths")
    if pl is not None:
        pl = pl.contiguous()
    toks = torch.zeros((B, T), dtype=torch.int32, device=pred.device)
    lens = torch.empty((B,), dtype=torch.int32, device=pred.device)
    lib = _lib.load()
    with _on_device(pred.device):
        rc = lib.ctcb_greedy_decode_typed(pred.data_ptr(), _DT_LOGITS[pred.dtype], pred.stride(ta), pred.stride(ba),
                                        pl.data_ptr() if pl is not None else None,
                                        _DT[pl.dtype] if pl is not None else 0, T, B, V, blank,
                                        -1 if unk is None else int(unk),
                                        toks.data_ptr(), lens.data_ptr(),
                                        _stream_ptr(pred.device))
    _lib.check(rc)
    return toks, lens


def edit_distance(ref, ref_lengths, hyp, hyp_lengths, totals=None):
    """Levenshtein distance of each (reference, hypothesis) row pair -- scripts/swbd/wer.py:45-68
    for a batch, on the device.  ref (B, Nmax) / hyp (B, Mmax) int32 CUDA tensors (unit stride
    along the row) with int32 lengths; ``greedy_decode``'s outputs can be passed as hyp/hyp_lengths.
    ``totals``: optional int64 CUDA tensor of 2, += {sum of distances, sum of reference lengths}.
    Returns (B,) int32."""
    for name, t in (("ref", ref), ("hyp", hyp), ("ref_lengths", ref_lengths), ("hyp_lengths", hyp_lengths)):
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise RuntimeError("edit_distance has no CPU path: %s must be a CUDA tensor" % name)
        if t.dtype != torch.int32:
            raise TypeError("%s must be int32, got %s" % (name, t.dtype))
    if ref.dim() != 2 or hyp.dim() != 2 or ref.shape[0] != hyp.shape[0]:
        raise ValueError("ref and hyp must be (B, N) and (B, M)")
    if ref.shape[1] > 1 and ref.stride(1) != 1:
        ref = ref.contiguous()
    if hyp.shape[1] > 1 and hyp.stride(1) != 1:
        hyp = hyp.contiguous()
    B = ref.shape[0]
    ref_lengths, hyp_lengths = ref_lengths.contiguous(), hyp_lengths.contiguous()
    if totals is not None and (totals.dtype != torch.int64 or totals.numel() < 2 or not totals.is_cuda):
        raise TypeError("totals must be an int64 CUDA tensor with two elements")
    out = torch.empty((B,), dtype=torch.int32, device=ref.device)
    with _on_device(ref.device):
        rc = _lib.load().ctcb_edit_distance(ref.data_ptr(), ref.stride(0), ref_lengths.data_ptr(),
                                            hyp.data_ptr(), hyp.stride(0), hyp_lengths.data_ptr(),
                                            B, ref.shape[1], hyp.shape[1], out.data_ptr(),
                                            totals.data_ptr() if totals is not None else None,
                                            _stream_ptr(ref.device))
    _lib.check(rc)
    return out
