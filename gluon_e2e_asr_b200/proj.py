"""The output projection fused with the CTC loss (SURVEY.md section 8f, rank 1).

Reference pair: ``self.tgt_proj(net_out)`` -- ``nn.Dense(units=V, flatten=False)``,
/root/reference/scripts/swbd/model.py:394-398 and :424 -- followed by
``loss_function(out, xpu_y, xpu_XL, xpu_yl)`` (train_ctc_ce.py:363, validation :143).
``proj_ctc_loss(hidden, weight, bias, label, ...)`` returns the same per-utterance losses as
``CtcLoss()(hidden @ weight.T + bias, label, ...)`` and is differentiable w.r.t. hidden, weight and bias.

The forward runs libctcb.so's ``ctcb_proj_forward``: a tcgen05 (tf32 in, fp32 accumulate in tensor memory) GEMM whose
epilogue produces what the lattice recursion reads; the logits are written once for the gradient kernel when a
gradient is needed and NOT AT ALL otherwise (``torch.no_grad()`` / validation).  The backward forms
d loss / d logits with ``ctcb_backward`` and then the three plain contractions (d hidden = G W, d weight = G^T hidden,
d bias = sum G) with torch.matmul -- library GEMMs, plumbing.  No CPU path.

``fused_training="recompute"`` trains without the logits: the forward keeps the lattice history and turns it into a
table of label-column occupancies (no logits buffer), and the backward's ``ctcb_proj_backward`` forms the product again
on the tensor cores and writes G directly from it -- the logits are never written or read.  The same three
contractions follow.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from .ops import _DT, _Call, _alloc_ws, _as_index_tensor, _blank_last, _on_device, _stream_ptr

__all__ = ["proj_ctc_loss", "proj_ctc_eval", "proj_greedy_decode", "ProjCtcLoss"]


def _proj_struct(hidden, weight, bias):
    pj = _lib.Proj()
    pj.hidden, pj.hidden_stride_b, pj.hidden_stride_t = hidden.data_ptr(), hidden.stride(0), hidden.stride(1)
    pj.K = hidden.shape[2]
    pj.weight = weight.data_ptr()
    pj.bias = bias.data_ptr() if bias is not None else None
    pj.operand_dtype = 1 if hidden.dtype == torch.bfloat16 else 0
    return pj


def _operands(hidden, weight, bias):
    """hidden, weight and bias checked and laid out as the projection kernel reads them (unit stride along K)."""
    for name, t in (("hidden", hidden), ("weight", weight)) + ((("bias", bias),) if bias is not None else ()):
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise RuntimeError("proj_ctc_loss has no CPU path: %s must be a CUDA tensor" % name)
    if hidden.dtype not in (torch.float32, torch.bfloat16) or weight.dtype != hidden.dtype:
        raise TypeError("hidden and weight must both be float32 (the reference's Dense dtype) or both bfloat16, got %s / %s"
                        % (hidden.dtype, weight.dtype))
    if bias is not None and bias.dtype != torch.float32:
        raise TypeError("bias must be float32, got %s" % bias.dtype)
    if hidden.dim() != 3 or weight.dim() != 2 or weight.shape[1] != hidden.shape[2]:
        raise ValueError("hidden must be (B, T, K) and weight (V, K)")
    if bias is not None and (bias.dim() != 1 or bias.shape[0] != weight.shape[0]):
        raise ValueError("bias must be (V,)")
    if hidden.stride(2) != 1:
        hidden = hidden.contiguous()
    return hidden, weight.contiguous(), bias.contiguous() if bias is not None else None


def _proj_problem(hidden, weight, logits, label, pred_lengths, label_lengths, blank_last, tn, need_grad):
    """The lattice problem of ``hidden @ weight.T``: ``(call, loss, ws, p)``.  ``logits``: the (B, T, V) fp32 buffer the
    forward writes, or None -- then the problem's logits pointer is NULL and only their shape is known."""
    B, T, _ = hidden.shape
    dev = hidden.device
    shape = logits if logits is not None else torch.empty((B, T, weight.shape[0]), dtype=torch.float32, device="meta")
    call = _Call(_MetaLogits(shape, dev), label, pred_lengths, label_lengths, blank_last, True, tn)
    loss = torch.empty((B,), dtype=torch.float32, device=dev)
    ws = _alloc_ws(call, need_grad)
    p = call.problem(loss)
    if logits is None:
        p.logits = None
    return call, loss, ws, p


class _tf32_matmul:
    """Library GEMMs of the training path at the precision of the fused product (tf32 in, fp32 accumulate)."""

    def __enter__(self):
        self.old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True

    def __exit__(self, *exc):
        torch.backends.cuda.matmul.allow_tf32 = self.old
        return False


class _ProjCtcLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, hidden, weight, bias, label, pred_lengths, label_lengths, blank_last, tn, fused=True):
        # fused: False (library product + CtcLoss), True (fused forward with a logits store) or "recompute"
        hidden, weight, bias = _operands(hidden, weight, bias)
        B, T, _ = hidden.shape
        dev = hidden.device
        need = any(ctx.needs_input_grad[:3])
        recompute = need and fused == "recompute"        # no logits: the backward forms the product again
        # the logits buffer exists only when a gradient will be asked for (NTC, like the model's output)
        if hidden.dtype == torch.bfloat16 and not recompute:
            fused = True              # no library GEMM gives fp32 logits from bfloat16 operands without a rounding in between
        if need and not fused:
            with _tf32_matmul():      # the library product, written once: what the gradient kernel reads
                logits = torch.nn.functional.linear(hidden, weight, bias)
        else:
            logits = torch.empty((B, T, weight.shape[0]), dtype=torch.float32, device=dev) if need and not recompute else None
        call, loss, ws, p = _proj_problem(hidden, weight, logits, label, pred_lengths, label_lengths, blank_last, tn, need)
        pj = _proj_struct(hidden, weight, bias)
        with _on_device(dev):
            if need and not fused:
                rc = _lib.load().ctcb_forward(ctypes.byref(p), 1, ws.data_ptr(), ws.numel(), _stream_ptr(dev))
            else:
                rc = _lib.load().ctcb_proj_forward(ctypes.byref(pj), ctypes.byref(p), 1 if need else 0, ws.data_ptr(), ws.numel(),
                                                   _stream_ptr(dev))
        _lib.check(rc)
        ctx.call, ctx.ws, ctx.logits = call, (ws if need else None), logits
        ctx.recompute = recompute
        ctx.save_for_backward(hidden, weight, bias)
        ctx.has_bias = bias is not None
        return loss

    @staticmethod
    def backward(ctx, head):
        hidden, weight, bias = ctx.saved_tensors
        call, ws, logits = ctx.call, ctx.ws, ctx.logits
        if ws is None:
            raise RuntimeError("proj_ctc_loss: backward needs a forward that ran with gradients enabled (and runs once)")
        head = head.to(torch.float32).contiguous()
        scratch = torch.empty((call.B,), dtype=torch.float32, device=head.device)
        if ctx.recompute:
            # the product again, straight into G: head * (softmax - occupancy), the logits never stored
            G = torch.empty((call.B, call.T, call.V), dtype=torch.float32, device=head.device)
            p = call.problem(scratch, grad=G, head=head)
            p.logits = None
            pj = _proj_struct(hidden, weight, bias)
            with _on_device(head.device):
                rc = _lib.load().ctcb_proj_backward(ctypes.byref(pj), ctypes.byref(p), ws.data_ptr(), ws.numel(),
                                                    _stream_ptr(head.device))
            _lib.check(rc)
        else:
            G = torch.empty_like(logits)
            call.data = logits
            call.run(_lib.PHASE_BACKWARD, ws, scratch, grad=G, head=head, handoff="pointer")
        ctx.ws = ctx.logits = None
        G2 = G.view(-1, G.shape[2])
        dh = dw = db = None
        with _tf32_matmul():
            if ctx.needs_input_grad[0]:
                dh = (G2 @ weight.float()).view(hidden.shape).to(hidden.dtype)
            if ctx.needs_input_grad[1]:
                dw = (G2.t() @ hidden.reshape(-1, hidden.shape[2]).float()).to(weight.dtype)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = G2.sum(0)
        return dh, dw, db, None, None, None, None, None, None


class _MetaLogits:
    """Shape / stride / device view of the logits tensor for _Call when the logits are never materialised."""

    def __init__(self, t, dev):
        self._t, self.device = t, dev
        self.shape = t.shape
        self.dtype = torch.float32          # the projection writes fp32 logits

    def stride(self, i):
        return self._t.stride(i)

    def data_ptr(self):
        return self._t.data_ptr() if self._t.device.type == "cuda" else 0


def proj_ctc_loss(hidden, weight, bias, label, pred_lengths=None, label_lengths=None, blank_label="first",
                  label_layout="NT", fused_training=False):
    """Per-utterance CTC loss (B,) of ``hidden (B,T,K) @ weight (V,K).T + bias`` -- model.py:424 + loss.py:121-139.

    tf32 tensor-core product (hidden and weight are read as they are; the low 13 mantissa bits do not take part),
    fp32 accumulation; everything after the product as in ``CtcLoss``.

    Without a gradient (validation, train_ctc_ce.py:143) the fused kernel runs and the logits never exist in HBM.
    With a gradient the logits have to exist for the gradient kernel; measured on B200 (scripts/proj_bench.py, cfg3
    shape, H = 512) a 2-SM 256x256 library GEMM writes them faster than the fused epilogue does (forward with logits
    kept: 211 us against 251), so by default the training call is the library product followed by ``CtcLoss``;
    ``fused_training=True`` forces the fused kernel (``ctcb_proj_forward`` with a logits buffer).

    ``fused_training="recompute"``: the fused forward without a logits buffer (it keeps a table of the label columns'
    occupancies instead), and a backward that forms the product again on the tensor cores and writes d loss / d logits
    straight from it (``ctcb_proj_backward``): the logits are never written or read.  Losses bit-identical to
    ``fused_training=True``; fp32 (tf32 product) or bfloat16 operands.  Measured against the other two arms in
    scripts/proj_train_bench.py (README)."""
    if isinstance(fused_training, str) and fused_training != "recompute":
        raise ValueError("fused_training must be False, True or 'recompute', got %r" % (fused_training,))
    needs_grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (hidden, weight, bias))
    fused = True if not needs_grad else (fused_training if fused_training == "recompute" else bool(fused_training))
    return _ProjCtcLossFn.apply(hidden, weight, bias, label, pred_lengths, label_lengths, _blank_last(blank_label),
                                label_layout == "TN", fused)


def proj_ctc_eval(hidden, weight, bias, label, pred_lengths=None, label_lengths=None, blank_label="first",
                  label_layout="NT", unk=None):
    """The validation pass from the encoder output (train_ctc_ce.py:143-160): ``(loss (B,), tokens (B,T) int32,
    lengths (B,) int32)`` of ``hidden @ weight.T + bias`` without the logits ever reaching HBM.

    ``loss`` is bit-identical to ``proj_ctc_loss`` under ``torch.no_grad()``.  ``tokens`` / ``lengths`` are
    ``greedy_decode(logits, pred_lengths, blank, unk=unk)`` of the logits the fused product forms (blank 0, or V - 1 for
    ``blank_label="last"``): the projection's epilogue keeps each frame's best two symbols while it reduces the row, and a
    small kernel collapses repeats and blanks.  The outputs go straight into ``edit_distance``.  fp32 (tf32 product) or
    bfloat16 operands; no autograd graph."""
    hidden, weight, bias = _operands(hidden, weight, bias)
    B, T, _ = hidden.shape
    dev = hidden.device
    _, loss, ws, p = _proj_problem(hidden, weight, None, label, pred_lengths, label_lengths, _blank_last(blank_label),
                                   label_layout == "TN", False)
    tokens = torch.empty((B, T), dtype=torch.int32, device=dev)
    lengths = torch.empty((B,), dtype=torch.int32, device=dev)
    pj = _proj_struct(hidden, weight, bias)
    with _on_device(dev):
        rc = _lib.load().ctcb_proj_forward_decode(ctypes.byref(pj), ctypes.byref(p), 0, -1 if unk is None else int(unk),
                                                  tokens.data_ptr(), lengths.data_ptr(), ws.data_ptr(), ws.numel(),
                                                  _stream_ptr(dev))
    _lib.check(rc)
    return loss, tokens, lengths


def proj_greedy_decode(hidden, weight, bias, pred_lengths=None, blank=0, unk=None):
    """Greedy decode from the encoder output without labels (decode_ctc.py:118-140: ``tgt_proj``, then the argmax with the
    ``<unk>`` rule): ``(tokens (B,T) int32, lengths (B,) int32)`` of ``hidden @ weight.T + bias``, the logits never stored.

    ``ctcb_proj_greedy_decode``: the projection's epilogue keeps each frame's best two symbols, a small kernel collapses
    repeats and ``blank``.  ``unk``: a frame whose best symbol is ``unk`` takes its second best (``greedy_decode``'s rule).
    Tokens and lengths are bit-identical to those of ``proj_ctc_eval`` for the same operands, lengths, blank and ``unk``,
    whatever its labels.  Any vocabulary size (no lattice, so no V > 64 condition).  fp32 (tf32 product) or bfloat16
    operands; no autograd graph.  The outputs go straight into ``edit_distance``."""
    hidden, weight, bias = _operands(hidden, weight, bias)
    B, T, _ = hidden.shape
    V = weight.shape[0]
    dev = hidden.device
    pl = _as_index_tensor(pred_lengths, dev, "pred_lengths")
    if pl is not None:
        if pl.dim() != 1 or pl.shape[0] != B:
            raise ValueError("pred_lengths must have shape (%d,)" % B)
        pl = pl.contiguous()
    tokens = torch.empty((B, T), dtype=torch.int32, device=dev)
    lengths = torch.empty((B,), dtype=torch.int32, device=dev)
    pj = _proj_struct(hidden, weight, bias)
    with _on_device(dev):
        rc = _lib.load().ctcb_proj_greedy_decode(ctypes.byref(pj), T, B, V, pl.data_ptr() if pl is not None else None,
                                                 _DT[pl.dtype] if pl is not None else 0, int(blank),
                                                 -1 if unk is None else int(unk), tokens.data_ptr(), lengths.data_ptr(),
                                                 _stream_ptr(dev))
    _lib.check(rc)
    return tokens, lengths


class ProjCtcLoss(torch.nn.Module):
    """``tgt_proj`` + ``CtcLoss`` as one block: holds the Dense parameters (units=V, in_units=K) in gluon's layout."""

    def __init__(self, in_units, units, use_bias=True, blank_label="first", label_layout="NT"):
        super().__init__()
        self.weight = torch.nn.Parameter(torch.empty(units, in_units))
        self.bias = torch.nn.Parameter(torch.zeros(units)) if use_bias else None
        torch.nn.init.uniform_(self.weight, -0.07, 0.07)
        self.blank_label, self.label_layout = blank_label, label_layout

    def forward(self, hidden, label, pred_lengths=None, label_lengths=None, fused_training=False):
        """``proj_ctc_loss`` with this block's parameters; ``fused_training``: False, True or "recompute" (see there)."""
        return proj_ctc_loss(hidden, self.weight, self.bias, label, pred_lengths, label_lengths, self.blank_label,
                             self.label_layout, fused_training)

    def evaluate(self, hidden, label, pred_lengths=None, label_lengths=None, unk=None):
        """``proj_ctc_eval`` with this block's parameters: (loss, tokens, lengths), the logits never stored."""
        return proj_ctc_eval(hidden, self.weight, self.bias, label, pred_lengths, label_lengths, self.blank_label,
                             self.label_layout, unk)

    def decode(self, hidden, pred_lengths=None, unk=None):
        """``proj_greedy_decode`` with this block's parameters and blank (0, or V - 1 for ``blank_label="last"``):
        (tokens, lengths) without labels, the logits never stored."""
        blank = self.weight.shape[0] - 1 if _blank_last(self.blank_label) else 0
        return proj_greedy_decode(hidden, self.weight, self.bias, pred_lengths, blank, unk)
