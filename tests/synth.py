"""Synthetic-input generator shared by tests and bench.py (SURVEY.md section 8d): the shapes
and dtypes the reference's data pipeline delivers -- float32 logits (B,T,V) in the model's NTC
layout (scripts/swbd/model.py:421-424), float32 0-padded labels (reader_kaldi_io.py:33-35,
train_ctc_ce.py:235), float32 lengths (gluonE2EASR/data/batchify.py:78-82)."""
import numpy as np

CONFIGS = {
    # name: (B, T, V, Lmax)   -- BASELINE.json "configs", in order
    "cfg1": (8, 200, 46, 50),
    "cfg2": (32, 500, 46, 120),
    "cfg3": (64, 500, 2000, 150),
    "cfg4": (16, 2000, 46, 300),
    "cfg5": (1024, 500, 46, 120),
}


def make_batch(B, T, V, L, seed=0, peaky=False, full_lengths=False, blank=0, scale=1.0):
    """Returns dict(pred (B,T,V) f32, label (B,L) f32 0-padded, pred_lengths (B,) f32,
    label_lengths (B,) f32).  Labels uniform over the non-blank symbols, L_b ~ U{ceil(L/2)..L}
    with one L_b = L, T_b ~ U{ceil(0.6T)..T} with one T_b = T, clamped feasible."""
    rng = np.random.Generator(np.random.PCG64(seed))
    lo, hi = (1, V) if blank == 0 else (0, V - 1)
    lab = rng.integers(lo, hi, (B, L))
    if full_lengths:
        Lb = np.full((B,), L)
        Tb = np.full((B,), T)
    else:
        Lb = rng.integers((L + 1) // 2, L + 1, B)
        Lb[rng.integers(0, B)] = L
        Tb = rng.integers(int(np.ceil(0.6 * T)), T + 1, B)
        Tb[rng.integers(0, B)] = T
    for b in range(B):
        rep = int((lab[b, 1:Lb[b]] == lab[b, :Lb[b] - 1]).sum()) if Lb[b] > 1 else 0
        Tb[b] = min(T, max(Tb[b], Lb[b] + rep))
        if Lb[b] + rep > Tb[b]:               # cannot be made feasible by T: shorten the label
            Lb[b] = max(0, Tb[b] // 2)
    x = (rng.standard_normal((B, T, V)) * scale).astype(np.float32)
    if peaky:
        for b in range(B):
            n, l = int(Tb[b]), int(Lb[b])
            if l == 0 or 2 * l > n:
                continue
            pos = np.sort(rng.choice(np.arange(0, n, 2), size=l, replace=False))
            path = np.full((n,), blank)
            path[pos] = lab[b, :l]
            x[b, np.arange(n), path] += 8.0
    labf = lab.astype(np.float32)
    for b in range(B):
        labf[b, Lb[b]:] = 0 if blank == 0 else -1
    return dict(pred=x, label=labf, pred_lengths=Tb.astype(np.float32),
                label_lengths=Lb.astype(np.float32))


# ---- inputs outside the documented ranges (the operator's parameter layer clamps them) -------------------------------
_BIG = {"f32": 3e9, "f64": 3e9, "i32": 2 ** 31 - 1, "i64": 2 ** 40}     # a length or label far beyond any T, Lmax, V
_NP = {"f32": np.float32, "f64": np.float64, "i32": np.int32, "i64": np.int64}


def _cast(vals, kind):
    """float64 master values -> dtype ``kind``: integer kinds get the truncated value, +-inf stands for that kind's big
    value (3e9 in floats, 2^31-1 in int32, 2^40 in int64; the labels' float one is 1e10)."""
    v = np.array(vals, np.float64)
    big = _BIG[kind]
    v = np.where(np.isinf(v), np.sign(v) * big, v)
    if kind in ("i32", "i64"):
        v = np.trunc(v)
    return v.astype(_NP[kind])


def hostile_batch(T, V, Lmax, blank_last=False, label_dtype="f32", length_dtype="f32", inferred=False, seed=0, rows=1):
    """One batch whose labels and lengths lie outside the ranges the operator documents, row by row:

    lengths: data_length > T, negative, fractional (x.9), == T, 0 and huge (2^40 / 3e9); label_length > Lmax, negative,
    fractional; labels >= V, negative, fractional, huge (1e10), equal to the blank at the first, middle and last
    position and twice in a row.  ``inferred``: no label lengths (rows end at the first padding value): a row without
    it (L = Lmax), a row that starts with it, and a row whose label truncates to it (-0.5 blank first, -1.5 blank last).
    Fractional values appear only in float dtypes (an integer dtype holds the truncated value).  Logits are N(0, 1):
    no frame comes near the emission floor.  ``rows`` > 1 repeats the hostile rows with fresh logits and labels.
    Returns dict(pred (B,T,V) f32, label (B,Lmax), pred_lengths (B,), label_lengths (B,) or None) as numpy arrays.
    """
    assert Lmax >= 8 and T >= 2 * Lmax + 4 and V >= 8
    rng = np.random.Generator(np.random.PCG64(seed))
    blank = V - 1 if blank_last else 0
    pad = -1.0 if blank_last else 0.0
    lo, hi = (0, V - 1) if blank_last else (1, V)
    inf = np.inf
    B0 = 18 if not inferred else 8
    B = B0 * rows
    lab = rng.integers(lo, hi, (B, Lmax)).astype(np.float64)
    for b in range(B):                                       # distinct neighbours: repeats only where a row puts them
        for j in range(1, Lmax):
            if lab[b, j] == lab[b, j - 1]:
                lab[b, j] = lo + (lab[b, j] - lo + 1) % (hi - lo)
    Tb = np.full((B,), float(T - 3))
    Lb = np.full((B,), float(Lmax // 2))
    lab_inf = np.zeros((B, Lmax), bool)                      # where the label is the dtype's big value
    for r in range(rows):
        o = r * B0
        if not inferred:
            Tb[o + 0] = T + 5                                # > T
            Tb[o + 1] = -3                                   # negative: 0 frames, infeasible
            Tb[o + 2] = T - 9.1                              # fractional (x.9): truncated, no status bit
            Tb[o + 3] = T; Lb[o + 3] = Lmax                  # == T, full label row
            Tb[o + 4] = 0                                    # no frames: infeasible
            Lb[o + 5] = Lmax + 7                             # > Lmax
            Lb[o + 6] = -2                                   # negative: empty label sequence
            Lb[o + 7] = 5.7                                  # fractional
            lab[o + 8, 1] = V; lab[o + 8, 3] = V + 3         # >= V
            lab[o + 9, 0] = -1; lab[o + 9, 2] = -7           # negative
            lab[o + 10, 1] = lo + 2.7; lab[o + 10, 2] = lo + 4.2   # fractional labels
            lab[o + 11, 0] = blank                           # label == blank: first, middle, last position
            lab[o + 11, Lmax // 4] = blank
            Lb[o + 11] = Lmax // 2; lab[o + 11, Lmax // 2 - 1] = blank
            lab[o + 12, 2] = blank; lab[o + 12, 3] = blank   # two adjacent labels == blank: a repeat
            Tb[o + 13] = inf                                 # huge length
            lab_inf[o + 13, 1] = True                        # huge label (1e10 / 2^31-1 / 2^40)
            Lb[o + 14] = inf                                 # huge label length
            lab[o + 15, 0] = lab[o + 15, 1] = V + 1          # two labels >= V: clamped to the same symbol, a repeat
            Tb[o + 16] = Lmax // 2; lab[o + 16, 2] = lab[o + 16, 3] = V + 2   # ... which makes this row infeasible
            Tb[o + 17] = -0.7                                # negative fraction: truncates to 0 (no clamp), infeasible
        else:
            Tb[o + 1] = T + 1                                # lengths are hostile here too
            lab[o + 1, 5] = pad                              # L = 5
            lab[o + 2, 0] = pad                              # starts with the padding value: L = 0
            lab[o + 3, 3] = pad - 0.5                        # truncates to the padding value: L = 3
            lab[o + 4, 2] = -7 if blank_last else V + 4      # a bad label (not the padding value) before the padding
            lab[o + 4, 6] = pad
            lab[o + 5, 1] = blank; lab[o + 5, 4] = pad       # label == blank inside the inferred length
            Tb[o + 6] = -2
            Tb[o + 7] = T - 0.5                              # row 0 of each group: no padding value, L = Lmax
    lbl = _cast(lab, label_dtype)
    if label_dtype in ("f32", "f64"):
        lbl[lab_inf] = 1e10
    else:
        lbl[lab_inf] = _BIG[label_dtype]
    x = rng.standard_normal((B, T, V)).astype(np.float32)
    return dict(pred=x, label=lbl, pred_lengths=_cast(Tb, length_dtype),
                label_lengths=None if inferred else _cast(Lb, length_dtype))
