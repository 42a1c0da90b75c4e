"""``CtcLoss`` -- the loss block the reference's training script instantiates.

Mirrors /root/reference/scripts/swbd/loss.py:54-139: same constructor arguments and
assertions (:111-119), same call signature ``(pred, label, pred_lengths=None,
label_lengths=None)`` -> ``(B,)`` (:121-139).  Differences, all inside the block:

* no ``swapaxes`` copies (:123-126): the kernels take the NTC / TN strides directly and
  write the gradient in the logits' own layout;
* the blank is index 0 (``blank_label='first'``) exactly as the reference hard-codes at :139
  -- its stale docstring (:74-76) and its ignored ``blank_label`` keyword (:122) are not
  followed.  ``blank_label='last'`` (upstream ``gluon.loss.CTCLoss``'s default) can be asked
  for at construction time.
"""
from __future__ import annotations

import torch

from . import ops

__all__ = ["CtcLoss"]


class CtcLoss(torch.nn.Module):
    def __init__(self, layout="NTC", label_layout="NT", weight=None, blank_label="first", **kwargs):
        assert layout in ["NTC", "TNC"], \
            "Only 'NTC' and 'TNC' layouts for pred are supported. Got: %s" % layout
        assert label_layout in ["NT", "TN"], \
            "Only 'NT' and 'TN' layouts for label are supported. Got: %s" % label_layout
        super().__init__()
        self._layout = layout
        self._label_layout = label_layout
        self._batch_axis = label_layout.find("N")
        self._weight = weight
        self._blank_label = blank_label
        ops._blank_last(blank_label)

    def forward(self, pred, label, pred_lengths=None, label_lengths=None, sample_weight=None):
        loss = ops._ctc_loss_layout(pred, label, pred_lengths, label_lengths, self._blank_label,
                                    self._layout, self._label_layout)
        # upstream gluon.loss.CTCLoss applies `weight` / `sample_weight`; the reference's block
        # takes neither, so they default to a no-op
        if self._weight is not None:
            loss = loss * self._weight
        if sample_weight is not None:
            loss = loss * sample_weight.reshape(-1)
        return loss

    hybrid_forward = forward   # name used by the reference (loss.py:121)

    def evaluate(self, pred, label, pred_lengths=None, label_lengths=None, unk=None):
        """The validation pass (train_ctc_ce.py:143-168) in one read of the logits: ``ops.ctc_eval`` with this block's
        layouts and blank -- ``(loss (B,), tokens (B,T) int32, lengths (B,) int32)``, the loss weighted as ``forward``
        weights it, no autograd graph.  ``tokens`` / ``lengths`` go straight into ``edit_distance``."""
        loss, tokens, lengths = ops.ctc_eval(pred, label, pred_lengths, label_lengths, self._blank_label, self._layout,
                                             self._label_layout, unk)
        if self._weight is not None:
            loss = loss * self._weight
        return loss, tokens, lengths

    def fused(self, pred, label, pred_lengths=None, label_lengths=None, head_grad=None, **kw):
        """loss and d(sum head*loss)/d pred in one library call (training hot path)."""
        return ops.ctc_loss_and_grad(pred, label, pred_lengths, label_lengths, head_grad,
                                     self._blank_label, self._layout, self._label_layout, **kw)
