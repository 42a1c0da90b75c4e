"""TEST INFRASTRUCTURE ONLY -- fp64 numpy restatement of the reference's CTC loss path.

This file is the *checker* for the CUDA path.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may import it.  Nothing under ``gluon_e2e_asr_b200/`` does.

What it restates
----------------
The reference computes its CTC training loss with one operator call

    scripts/swbd/loss.py:134-139   F.contrib.ctc_loss(data, label, data_lengths,
                                       label_lengths, use_data_lengths,
                                       use_label_lengths, blank_label='first')

wrapped by ``CtcLoss.hybrid_forward`` (scripts/swbd/loss.py:121-139: the NTC->TNC
``swapaxes`` at :123-124 and the TN->NT label swap at :125-126) and called from
scripts/swbd/train_ctc_ce.py:143 and :363.  The arithmetic lives in Apache MXNet 1.x
(``_contrib_ctc_loss`` -> vendored Baidu warp-ctc), which is NOT vendored in
/root/reference and is NOT installable in this image.  The reference pins no MXNet
version (no requirements/setup file; scripts/swbd/loss.py only needs the
``blank_label`` keyword, i.e. MXNet >= 1.3).  This module therefore restates the
*published* algorithm (Graves et al. 2006 as realised by warp-ctc, SURVEY.md
Appendix A) and is pinned by

  * upstream MXNet / warp-ctc known-answer vectors K1-K5 (SURVEY.md section 4),
    see tests/golden/kat.json and tests/test_oracle.py;
  * torch's independent CPU ``ctc_loss`` in fp64 (tests/test_oracle.py);
  * fp64 finite differences of the loss (tests/test_oracle.py).

PARITY STATUS: "parity unpinned by the reference itself" -- the reference holds no
tests, golden vectors or fixtures for this path (SURVEY.md section 4); the pins
above are upstream's, recalled and numerically re-verified.

Everything is computed in log space in float64; the gradient uses the per-frame
identity  sum_s alpha_t(s) beta_t(s) / y_t(ext_s) = P  so it never subtracts two
large log-likelihoods.
"""
from __future__ import annotations

import numpy as np

__all__ = [
    "infer_lengths",
    "param_layer",
    "ctc_loss_grad",
    "ctc_loss_op",
    "CtcLossOracle",
    "greedy_decode",
    "split_and_load_slices",
]

NEG_INF = -np.inf


def _logsumexp(a, axis=None):
    m = np.max(a, axis=axis, keepdims=True)
    m = np.where(np.isfinite(m), m, 0.0)
    with np.errstate(divide="ignore"):
        out = np.log(np.sum(np.exp(a - m), axis=axis, keepdims=True)) + m
    return np.squeeze(out, axis=axis) if axis is not None else out.reshape(())


def infer_lengths(label, data_lengths, label_lengths, T, use_data_lengths,
                  use_label_lengths, blank_label="first"):
    """Length semantics of the operator's parameter layer (SURVEY.md section 8 row a3).

    * ``use_data_lengths``  False -> every utterance has T frames; True -> trunc(data_lengths).
    * ``use_label_lengths`` False -> length = index of the first padding value in the
      label row (0 for blank_label='first', -1 for 'last'), or Lmax if none;
      True -> trunc(label_lengths).
    The reference always passes both (scripts/swbd/train_ctc_ce.py:143, :363) as float32
    (gluonE2EASR/data/batchify.py:78-82), hence the truncation.
    """
    label = np.asarray(label)
    B, Lmax = label.shape
    if use_data_lengths:
        T_b = _trunc(data_lengths)
    else:
        T_b = np.full((B,), T, dtype=np.int64)
    if use_label_lengths:
        L_b = _trunc(label_lengths)
    else:
        pad = 0 if blank_label == "first" else -1
        is_pad = _trunc(label) == pad
        L_b = np.where(is_pad.any(axis=1), is_pad.argmax(axis=1), Lmax).astype(np.int64)
    return T_b, L_b


UTT_INFEASIBLE, UTT_BAD_LABEL, UTT_LEN_CLAMPED = 1, 2, 4


def _trunc(a):
    """Truncation toward zero to int64, like the operator's cast (integers pass unchanged)."""
    a = np.asarray(a)
    if a.dtype.kind in "iu":
        return a.astype(np.int64)
    return np.trunc(a.astype(np.float64)).astype(np.int64)


def param_layer(label, data_lengths, label_lengths, T, V, blank_label="first"):
    """The operator's parameter layer: what the lattice kernels make of the caller's labels and lengths.

    label (B, Lmax) of any numeric dtype; ``data_lengths`` / ``label_lengths`` (B,) or None (= T, resp. the
    index of the first padding value -- 0 for blank_label='first', -1 for 'last' -- or Lmax).  Contract:

    * lengths are truncated toward zero and clamped to [0, T] and [0, Lmax]; CTCB_UTT_LEN_CLAMPED (4) when a
      clamp changed the truncated value (a fractional length sets nothing);
    * an inferred label length compares the truncated, *unclamped* label with the padding value;
    * labels are truncated toward zero and clamped to [0, V-1]; CTCB_UTT_BAD_LABEL (2) when one of the first
      L_b truncated labels was < 0, >= V or equal to the blank (such a label is a lattice state of its own);
    * CTCB_UTT_INFEASIBLE (1) when T_b == 0 or L_b + repeats > T_b (repeats of the clamped labels).

    Returns (T_b, L_b, labels, status): int64 (B,), int64 (B,), int64 (B, Lmax) clamped, int32 (B,) without
    CTCB_UTT_WIDE_LOGITS (8), which depends on the logits.
    """
    raw = _trunc(label)
    B, Lmax = raw.shape
    blank = 0 if blank_label == "first" else V - 1
    status = np.zeros((B,), np.int32)
    if data_lengths is None:
        T_b = np.full((B,), T, np.int64)
    else:
        t = _trunc(data_lengths)
        T_b = np.clip(t, 0, T)
        status |= np.where(T_b != t, UTT_LEN_CLAMPED, 0).astype(np.int32)
    if label_lengths is None:
        _, L_b = infer_lengths(raw, None, None, T, False, False, blank_label)
    else:
        l = _trunc(label_lengths)
        L_b = np.clip(l, 0, Lmax)
        status |= np.where(L_b != l, UTT_LEN_CLAMPED, 0).astype(np.int32)
    lab = np.clip(raw, 0, V - 1)
    for b in range(B):
        r = raw[b, :L_b[b]]
        if np.any((r < 0) | (r >= V) | (r == blank)):
            status[b] |= UTT_BAD_LABEL
        c = lab[b, :L_b[b]]
        repeats = int(np.sum(c[1:] == c[:-1])) if L_b[b] > 1 else 0
        if T_b[b] <= 0 or L_b[b] + repeats > T_b[b]:
            status[b] |= UTT_INFEASIBLE
    return T_b, L_b, lab, status


def _one_utterance(x, lab, blank):
    """x: (T_b, V) float64 logits of the valid frames; lab: (L,) int labels.

    Returns (loss, G) with G = d loss / d x, shape (T_b, V).  Spec: SURVEY.md
    Appendix A (alpha/beta over ext = [blank, l1, blank, ..., lL, blank]).
    """
    Tb, V = x.shape
    L = int(lab.shape[0])
    S = 2 * L + 1
    logy = x - _logsumexp(x, axis=1)[:, None]           # log softmax, (T_b, V)
    y = np.exp(logy)

    ext = np.full((S,), blank, dtype=np.int64)
    ext[1::2] = lab
    # s-2 -> s transition allowed exactly when the two symbols differ.  Even states are blanks (never); a label
    # state j skips in when label j != label j-1 -- a label equal to the blank is a state of its own (torch's rule;
    # warp-ctc also forbids the skip into it, which can leave an utterance of L + repeats <= T_b without a path)
    skip = np.zeros((S,), dtype=bool)
    if S > 2:
        skip[2:] = ext[2:] != ext[:-2]
    repeats = int(np.sum(lab[1:] == lab[:-1])) if L > 1 else 0
    if Tb <= 0 or L + repeats > Tb:
        # infeasible alignment: defined behaviour = cost 0, gradient 0 (SURVEY.md 7.3-6,
        # warp-ctc's behaviour); torch returns +inf here.
        return 0.0, np.zeros_like(x), False

    em = logy[:, ext]                                   # (T_b, S) emissions along the lattice

    def shift(a, k):
        out = np.full_like(a, NEG_INF)
        out[k:] = a[:-k] if k else a
        return out

    alpha = np.full((Tb, S), NEG_INF)
    alpha[0, 0] = em[0, 0]
    if S > 1:
        alpha[0, 1] = em[0, 1]
    for t in range(1, Tb):
        p = alpha[t - 1]
        stack = np.stack([p, shift(p, 1), np.where(skip, shift(p, 2), NEG_INF)])
        alpha[t] = em[t] + _logsumexp(stack, axis=0)
    tail = alpha[Tb - 1, S - 1:S] if S == 1 else alpha[Tb - 1, S - 2:S]
    loglik = float(_logsumexp(tail, axis=0))

    # beta_t(s) includes the emission at t (mirrors alpha)
    def shiftl(a, k):
        out = np.full_like(a, NEG_INF)
        out[:-k] = a[k:]
        return out

    skip_out = np.zeros((S,), dtype=bool)               # s -> s+2 allowed
    if S > 2:
        skip_out[:-2] = skip[2:]
    beta = np.full((Tb, S), NEG_INF)
    beta[Tb - 1, S - 1] = em[Tb - 1, S - 1]
    if S > 1:
        beta[Tb - 1, S - 2] = em[Tb - 1, S - 2]
    for t in range(Tb - 2, -1, -1):
        n = beta[t + 1]
        stack = np.stack([n, shiftl(n, 1), np.where(skip_out, shiftl(n, 2), NEG_INF)])
        beta[t] = em[t] + _logsumexp(stack, axis=0)

    # posterior state occupancy, normalised per frame (sum_s == 1 analytically)
    lg = alpha + beta - em
    lg = lg - _logsumexp(lg, axis=1)[:, None]
    gamma = np.exp(lg)                                  # (T_b, S)
    occ = np.zeros((Tb, V))
    np.add.at(occ, (np.arange(Tb)[:, None], ext[None, :]), gamma)
    G = y - occ
    return -loglik, G, True


def ctc_loss_grad(data_tbv, label, T_b, L_b, blank=0, head_grad=None):
    """Per-utterance loss (B,) and d(sum_b head[b] loss[b])/d data, TNC layout.

    data_tbv : (T, B, V) logits (unnormalised; the softmax is inside the op).
    label    : (B, Lmax) any numeric dtype, truncated to int (reader_kaldi_io.py:33-35
               delivers float32 labels) and clamped to [0, V-1].
    Padded frames t >= T_b[b] get gradient 0 (SURVEY.md section 0 fact 6).
    Returns (loss, grad, feasible) as float64 / bool arrays.
    """
    x = np.asarray(data_tbv, dtype=np.float64)
    T, B, V = x.shape
    lab = np.clip(_trunc(label), 0, V - 1)
    loss = np.zeros((B,))
    grad = np.zeros_like(x)
    ok = np.zeros((B,), dtype=bool)
    head = np.ones((B,)) if head_grad is None else np.asarray(head_grad, dtype=np.float64)
    for b in range(B):
        tb = int(min(max(int(T_b[b]), 0), T))
        lb = int(min(max(int(L_b[b]), 0), lab.shape[1]))
        l, g, f = _one_utterance(x[:tb, b, :], lab[b, :lb], blank)
        loss[b] = l
        grad[:tb, b, :] = head[b] * g
        ok[b] = f
    return loss, grad, ok


def ctc_loss_op(data, label, data_lengths=None, label_lengths=None,
                use_data_lengths=False, use_label_lengths=False, blank_label="first",
                head_grad=None):
    """The raw operator surface ``mx.nd.contrib.ctc_loss`` as the reference calls it
    (scripts/swbd/loss.py:134-139).  data is TNC.  Returns (loss, grad_tnc, feasible)."""
    data = np.asarray(data)
    T, B, V = data.shape
    assert blank_label in ("first", "last")
    blank = 0 if blank_label == "first" else V - 1
    T_b, L_b, lab, _ = param_layer(label, data_lengths if use_data_lengths else None,
                                   label_lengths if use_label_lengths else None, T, V, blank_label)
    return ctc_loss_grad(data, lab, T_b, L_b, blank=blank, head_grad=head_grad)


class CtcLossOracle:
    """``CtcLoss(layout, label_layout)`` of scripts/swbd/loss.py:111-139, restated.

    The reference hard-codes blank_label='first' at loss.py:139 (the hybrid_forward
    keyword of the same name at :122 is ignored); upstream ``gluon.loss.CTCLoss``
    defaults to 'last'.  ``blank_label`` here is a constructor argument so both can be
    checked; the default follows the reference.
    """

    def __init__(self, layout="NTC", label_layout="NT", blank_label="first"):
        assert layout in ("NTC", "TNC"), layout
        assert label_layout in ("NT", "TN"), label_layout
        self.layout, self.label_layout, self.blank_label = layout, label_layout, blank_label

    def __call__(self, pred, label, pred_lengths=None, label_lengths=None, head_grad=None):
        pred = np.asarray(pred)
        label = np.asarray(label)
        if self.layout == "NTC":
            pred = np.swapaxes(pred, 0, 1)              # loss.py:123-124
        if self.label_layout == "TN":
            label = np.swapaxes(label, 0, 1)            # loss.py:125-126
        loss, g, ok = ctc_loss_op(pred, label, pred_lengths, label_lengths,
                                  use_data_lengths=pred_lengths is not None,
                                  use_label_lengths=label_lengths is not None,
                                  blank_label=self.blank_label, head_grad=head_grad)
        if self.layout == "NTC":
            g = np.swapaxes(g, 0, 1)
        return loss, g, ok


def _clamped_length(lengths, b, T):
    """Frame count of utterance b: truncated toward zero, clamped to [0, T] (as the decode kernel does)."""
    return int(min(max(int(_trunc(np.asarray(lengths)[b])), 0), T))


def greedy_decode(logits_btv, lengths, blank=0):
    """Greedy CTC decode of scripts/swbd/train_ctc_ce.py:149-160: argmax over V, collapse
    repeats, drop blank (index 0).  Returns a list of int lists."""
    logits = np.asarray(logits_btv)
    out = []
    for b in range(logits.shape[0]):
        n = _clamped_length(lengths, b, logits.shape[1])
        path = np.argmax(logits[b, :n], axis=1)
        seq, prev = [], None
        for j, c in enumerate(path):
            c = int(c)
            if j == 0 or c != prev:
                if c != blank:
                    seq.append(c)
            prev = c
        out.append(seq)
    return out


def greedy_decode_unk(logits_btv, lengths, unk, blank=0):
    """Greedy decode with the ``<unk>`` rule of scripts/swbd/decode_ctc.py:120-140, restated loop for
    loop: ``trans``/``trans2`` are the best and second best symbol of every frame (descending argsort,
    :125-127; ties here: lowest index first); ``prev = trans[j-1]`` is the RAW best symbol of the
    previous frame (:133), ``curr = trans[j]`` or ``trans2[j]`` when ``trans[j] == unk`` (:134-136); the
    symbol is emitted when ``j == 0 or curr != prev`` and it is not the blank (:138-140)."""
    logits = np.asarray(logits_btv)
    out = []
    for b in range(logits.shape[0]):
        n = _clamped_length(lengths, b, logits.shape[1])
        order = np.argsort(-logits[b, :n], axis=1, kind="stable")
        trans, trans2 = order[:, 0], order[:, 1] if logits.shape[2] > 1 else order[:, 0]
        seq = []
        for j in range(n):
            prev = int(trans[j - 1])
            curr = int(trans[j])
            if curr == unk:
                curr = int(trans2[j])
            if j == 0 or curr != prev:
                if curr != blank:
                    seq.append(curr)
        out.append(seq)
    return out


def split_and_load_slices(n, k):
    """Batch-axis slices of scripts/swbd/utils.py:25-33 (``split_and_load``): k-1 chunks of
    n//k, the remainder on the last device; if n < k everything goes to device 0."""
    if n < k:
        return [slice(0, n)]
    m = n // k
    return [slice(i * m, (i + 1) * m) for i in range(k - 1)] + [slice((k - 1) * m, n)]


def edit_distance(ref, hyp):
    """scripts/swbd/wer.py:45-68 (`_edit_distance`): full (N+1) x (M+1) table; a match copies the
    diagonal, otherwise 1 + the smallest of the three neighbours."""
    n, m = len(ref), len(hyp)
    tab = [[0] * (m + 1) for _ in range(n + 1)]
    for i in range(n + 1):
        tab[i][0] = i
    for j in range(m + 1):
        tab[0][j] = j
    for i in range(1, n + 1):
        for j in range(1, m + 1):
            if ref[i - 1] == hyp[j - 1]:
                tab[i][j] = tab[i - 1][j - 1]
            else:
                tab[i][j] = 1 + min(tab[i - 1][j], tab[i][j - 1], tab[i - 1][j - 1])
    return tab[n][m]


def compute_wer(reference_corpus, translation_corpus, lower_case=False):
    """scripts/swbd/wer.py:9-43: total edit distance over total reference length."""
    dist = words = 0
    for ref, hyp in zip(reference_corpus, translation_corpus):
        if lower_case:
            ref, hyp = [w.lower() for w in ref], [w.lower() for w in hyp]
        dist += edit_distance(ref, hyp)
        words += len(ref)
    return dist / words
