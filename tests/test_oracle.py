"""CPU tests of the oracle itself: oracle/ctc_oracle.py (numpy fp64) and oracle/ctc_ref.c
(C restatement, fp32 + fp64) against the committed golden vectors (upstream KATs K1-K5,
torch-fp64 fixtures), closed forms, finite differences and each other."""
import json
import os

import numpy as np
import pytest

from oracle import ctc_oracle as O
from oracle import ctc_ref as R
from tests.synth import make_batch


def _kats(golden_dir):
    with open(os.path.join(golden_dir, "kat.json")) as f:
        return json.load(f)


def test_kat_numpy_oracle(golden_dir):
    for k in _kats(golden_dir):
        orc = O.CtcLossOracle(layout=k["layout"], label_layout="NT", blank_label=k["blank_label"])
        loss, _, ok = orc(np.array(k["data"], np.float32), np.array(k["label"]))
        assert ok.all()
        np.testing.assert_allclose(loss, k["expect"], rtol=k["rtol"], err_msg=k["name"])


def test_kat_k4_variants(golden_dir):
    k = [k for k in _kats(golden_dir) if k["name"].startswith("K4")][0]
    data = np.array(k["data"], np.float32)
    lab = np.array(k["label"])
    exp = np.array(k["expect"])
    ntc = O.CtcLossOracle("NTC", "NT", "last")
    tnc = O.CtcLossOracle("TNC", "NT", "last")
    tn = O.CtcLossOracle("NTC", "TN", "last")
    np.testing.assert_allclose(tnc(data.swapaxes(0, 1), lab)[0], exp, rtol=2e-7)
    np.testing.assert_allclose(tn(data, lab.T)[0], exp, rtol=2e-7)
    np.testing.assert_allclose(ntc(data, lab, None, np.array([2, 3]))[0], exp, rtol=2e-7)
    np.testing.assert_allclose(ntc(data, lab, np.array([20, 20]), np.array([2, 3]))[0], exp, rtol=2e-7)
    # shorter pred_lengths change the answer and only read the first frames
    a = ntc(data, lab, np.array([10, 10]), np.array([2, 3]))[0]
    b = ntc(data[:, :10], lab, None, np.array([2, 3]))[0]
    np.testing.assert_allclose(a, b, rtol=1e-12)


def test_kat_c_port(golden_dir):
    for k in _kats(golden_dir):
        data = np.array(k["data"], np.float64)
        if k["layout"] == "NTC":
            data = data.swapaxes(0, 1)
        lab = np.array(k["label"])
        T = data.shape[0]
        V = data.shape[2]
        blank = 0 if k["blank_label"] == "first" else V - 1
        Tb, Lb = O.infer_lengths(lab, None, None, T, False, False, k["blank_label"])
        for dt, rt in ((np.float64, k["rtol"]), (np.float32, max(k["rtol"], 2e-6))):
            loss, _, ok = R.ctc_ref(data, lab, Tb, Lb, blank=blank, dtype=dt)
            assert ok.all()
            np.testing.assert_allclose(loss, k["expect"], rtol=rt, err_msg=k["name"])


def _golden_cases(golden_dir):
    z = np.load(os.path.join(golden_dir, "torch_fp64.npz"))
    names = sorted({k.split("/")[0] for k in z.files})
    return [(n, {k.split("/")[1]: z[k] for k in z.files if k.startswith(n + "/")}) for n in names]


def test_torch_fp64_fixtures_numpy_and_c(golden_dir):
    for name, c in _golden_cases(golden_dir):
        blank = int(c["blank"])
        loss, grad, ok = O.ctc_loss_grad(c["data"], c["label"], c["T_b"], c["L_b"], blank, c["head"])
        assert ok.all(), name
        np.testing.assert_allclose(loss, c["loss"], rtol=1e-12, atol=1e-12, err_msg=name)
        np.testing.assert_allclose(grad, c["grad"], rtol=1e-10, atol=1e-12, err_msg=name)
        l2, g2, ok2 = R.ctc_ref(c["data"], c["label"], c["T_b"], c["L_b"], blank, c["head"], dtype=np.float64)
        assert ok2.all()
        np.testing.assert_allclose(l2, c["loss"], rtol=1e-11, atol=1e-11, err_msg=name)
        np.testing.assert_allclose(g2, c["grad"], rtol=1e-8, atol=1e-11, err_msg=name)


def test_closed_forms():
    rng = np.random.default_rng(7)
    T, V = 9, 6
    x = rng.standard_normal((T, 1, V))
    logy = x - np.log(np.exp(x).sum(-1, keepdims=True))
    # L = 0: the only path is all blanks
    loss, g, ok = O.ctc_loss_grad(x, np.zeros((1, 1)), [T], [0])
    np.testing.assert_allclose(loss[0], -logy[:, 0, 0].sum(), rtol=1e-13)
    # T == L, no repeats: single path
    lab = np.array([[1, 2, 3, 4, 5, 1, 2, 3, 4]])
    loss, g, ok = O.ctc_loss_grad(x, lab, [T], [T])
    np.testing.assert_allclose(loss[0], -logy[np.arange(T), 0, lab[0]].sum(), rtol=1e-13)
    # single-path gradient: softmax - onehot
    y = np.exp(logy[:, 0])
    oh = np.zeros_like(y); oh[np.arange(T), lab[0]] = 1
    np.testing.assert_allclose(g[:, 0], y - oh, atol=1e-13)


def test_infeasible_defined_behaviour():
    x = np.random.default_rng(0).standard_normal((3, 2, 5))
    lab = np.array([[1, 1, 2], [1, 2, 3]])        # row 0 needs 4 frames (one repeat), row 1 fits
    loss, g, ok = O.ctc_loss_grad(x, lab, [3, 3], [3, 3])
    assert list(ok) == [False, True]
    assert loss[0] == 0 and np.all(g[:, 0] == 0) and loss[1] > 0
    l2, g2, ok2 = R.ctc_ref(x, lab, [3, 3], [3, 3], dtype=np.float64)
    assert list(ok2) == [False, True] and l2[0] == 0 and np.all(g2[:, 0] == 0)


def test_finite_difference_gradient():
    rng = np.random.default_rng(3)
    T, B, V, L = 7, 2, 5, 3
    x = rng.standard_normal((T, B, V))
    lab = np.array([[1, 1, 2], [3, 4, 0]])
    Tb, Lb = np.array([7, 5]), np.array([3, 2])
    head = np.array([0.7, 1.3])
    _, g, _ = O.ctc_loss_grad(x, lab, Tb, Lb, head_grad=head)
    eps = 1e-6
    num = np.zeros_like(x)
    for idx in np.ndindex(*x.shape):
        xp = x.copy(); xp[idx] += eps
        xm = x.copy(); xm[idx] -= eps
        lp = (O.ctc_loss_grad(xp, lab, Tb, Lb)[0] * head).sum()
        lm = (O.ctc_loss_grad(xm, lab, Tb, Lb)[0] * head).sum()
        num[idx] = (lp - lm) / (2 * eps)
    np.testing.assert_allclose(g, num, atol=2e-8)
    assert np.all(g[5:, 1] == 0)                 # padded frames


def test_properties_batch_vs_single_and_row_sums():
    d = make_batch(6, 40, 11, 9, seed=5)
    x = d["pred"].swapaxes(0, 1)
    Tb, Lb = d["pred_lengths"], d["label_lengths"]
    loss, g, ok = O.ctc_loss_grad(x, d["label"], Tb, Lb)
    assert ok.all()
    for b in range(6):
        l1, g1, _ = O.ctc_loss_grad(x[:, b:b + 1], d["label"][b:b + 1], Tb[b:b + 1], Lb[b:b + 1])
        np.testing.assert_allclose(l1[0], loss[b], rtol=1e-13)
        np.testing.assert_allclose(g1[:, 0], g[:, b], atol=1e-14)
        np.testing.assert_allclose(g[:int(Tb[b]), b].sum(-1), 0, atol=1e-12)   # sum_v G = 0
        assert np.all(g[int(Tb[b]):, b] == 0)


def test_length_inference():
    lab = np.array([[3, 2, 0, 0], [1, 2, 3, 4], [0, 0, 0, 0]], np.float32)
    Tb, Lb = O.infer_lengths(lab, None, None, 10, False, False, "first")
    assert list(Tb) == [10, 10, 10] and list(Lb) == [2, 4, 0]
    lab2 = np.array([[3, 0, -1, -1], [-1, 2, 3, 4]], np.float32)
    assert list(O.infer_lengths(lab2, None, None, 5, False, False, "last")[1]) == [2, 0]
    Tb, Lb = O.infer_lengths(lab, np.array([3.9, 2.0, 7.0], np.float32), np.array([1.0, 3.2, 0.0]), 10, True, True)
    assert list(Tb) == [3, 2, 7] and list(Lb) == [1, 3, 0]


def test_c_fp32_port_is_reference_class_not_oracle():
    """The fp32 port reproduces the log-space fp32 error the survey measured (SURVEY.md 7.3-1):
    close in loss (relative), far outside rtol 1e-4/atol 1e-5 on the gradient at cfg2 size."""
    d = make_batch(4, 500, 46, 120, seed=0)
    x = d["pred"].swapaxes(0, 1)
    lo, go, _ = O.ctc_loss_grad(x, d["label"], d["pred_lengths"], d["label_lengths"])
    l32, g32, _ = R.ctc_ref(x, d["label"], d["pred_lengths"], d["label_lengths"], dtype=np.float32)
    np.testing.assert_allclose(l32, lo, rtol=1e-5)
    assert np.abs(g32 - go).max() < 2e-2


def test_greedy_decode_and_split():
    logits = np.zeros((1, 6, 4)); path = [0, 2, 2, 0, 2, 3]
    logits[0, np.arange(6), path] = 5
    assert O.greedy_decode(logits, [6]) == [[2, 2, 3]]
    assert O.greedy_decode(logits, [3]) == [[2]]
    s = O.split_and_load_slices(10, 4)
    assert [(x.start, x.stop) for x in s] == [(0, 2), (2, 4), (4, 6), (6, 10)]
    assert [(x.start, x.stop) for x in O.split_and_load_slices(3, 4)] == [(0, 3)]


def test_c_fp64_matches_numpy_at_size():
    """The C restatement in fp64 is the checker of the full-batch-size GPU parity tests
    (tests/test_parity_gpu.py::test_baseline_configs_at_full_batch_size): pin it to the numpy oracle
    on BASELINE-shaped utterances (NTC strides, ragged lengths, repeats, head gradient, peaky logits)."""
    for seed, peaky, shape in ((5, True, (6, 300, 46, 80)), (6, False, (4, 500, 46, 120)), (7, False, (2, 120, 300, 40))):
        d = make_batch(*shape, seed=seed, peaky=peaky)
        head = np.random.default_rng(seed).uniform(0.5, 1.5, shape[0])
        lo, go, ok = O.CtcLossOracle("NTC", "NT")(d["pred"], d["label"], d["pred_lengths"], d["label_lengths"], head_grad=head)
        lc, gc, okc = R.ctc_ref(d["pred"], d["label"], d["pred_lengths"], d["label_lengths"], head_grad=head,
                                layout="NTC", dtype=np.float64)
        assert ok.all() and okc.all()
        np.testing.assert_allclose(lc, lo, rtol=1e-12, atol=1e-11)
        np.testing.assert_allclose(gc, go, rtol=1e-9, atol=1e-12)


def test_greedy_decode_unk_rule():
    """decode_ctc.py:120-140 restated: <unk> -> second best; `prev` stays the raw best of the previous frame."""
    unk = 3
    x = np.zeros((1, 7, 5))
    #        best:  2    unk(2nd 2)  unk(2nd 1)  1    0(blank)  unk(2nd 0)  4
    best = [2, unk, unk, 1, 0, unk, 4]
    second = [1, 2, 1, 2, 1, 0, 2]
    for j, (a, b) in enumerate(zip(best, second)):
        x[0, j, a] = 5.0; x[0, j, b] = 4.0
    # j=1: curr=2 vs prev=2 (raw) -> dropped; j=2: curr=1 vs prev=unk -> kept; j=3: curr=1 vs prev=unk -> kept (the
    # reference compares with the RAW previous symbol, so the repeated 1 is NOT collapsed); j=5: curr=0 blank dropped
    assert O.greedy_decode_unk(x, [7], unk) == [[2, 1, 1, 4]]
    assert O.greedy_decode_unk(x, [7], -1) == O.greedy_decode(x, [7])


# ---- the parameter layer: labels equal to the blank, out-of-range labels, clamped lengths -----------------------------
def _torch_fp64_loss(x_tbv, lab, Tb, Lb, blank):
    """torch's CPU ctc_loss in fp64 (an independent restatement of the forward), per utterance."""
    torch = pytest.importorskip("torch")
    xt = torch.tensor(x_tbv, dtype=torch.float64)
    return torch.nn.functional.ctc_loss(xt.log_softmax(-1), torch.tensor(lab, dtype=torch.long),
                                        torch.tensor(Tb, dtype=torch.long), torch.tensor(Lb, dtype=torch.long),
                                        blank=blank, reduction="none", zero_infinity=False).numpy()


@pytest.mark.parametrize("blank_last", [False, True])
def test_label_equal_to_blank_matches_torch_fp64(blank_last):
    """A label equal to the blank is a lattice state of its own that emits with the blank's probability, and the skip
    into label j is allowed exactly when label j != label j-1 (torch's rule).  Both oracles agree with torch's fp64
    ctc_loss on rows with such labels at the first, middle and last position, twice in a row, and with only L + repeats
    frames -- where forbidding the skip into it (warp-ctc's rule) leaves no path at all and an infinite loss.

    The gradients are checked against central differences of torch's loss: torch's own backward is wrong when the
    LAST label equals the blank (it does not match the derivative of its forward there)."""
    rng = np.random.default_rng(31)
    T, V = 9, 6
    bl = V - 1 if blank_last else 0
    a, c = (1, 2) if not blank_last else (0, 2)
    rows = [([a, bl, c], 6), ([bl, a, bl], 7), ([a, bl, bl], 4), ([bl, bl, bl], 5), ([c, a, bl], 9),
            ([a, c, a], 3), ([bl, c, c], 5)]
    B, L = len(rows), 3
    lab = np.array([r for r, _ in rows], np.int64)
    Tb = np.array([t for _, t in rows], np.int64)
    Lb = np.full((B,), L, np.int64)
    x = rng.standard_normal((T, B, V))
    head = rng.uniform(0.5, 1.5, B)
    lt = _torch_fp64_loss(x, lab, Tb, Lb, bl)
    assert np.isfinite(lt).all()
    eps = 1e-6
    gt = np.zeros_like(x)
    for idx in np.ndindex(*x.shape):
        xp = x.copy(); xp[idx] += eps
        xm = x.copy(); xm[idx] -= eps
        gt[idx] = ((_torch_fp64_loss(xp, lab, Tb, Lb, bl) - _torch_fp64_loss(xm, lab, Tb, Lb, bl)) * head).sum() / (2 * eps)
    lo, go, ok = O.ctc_loss_grad(x, lab, Tb, Lb, bl, head)
    lc, gc, okc = R.ctc_ref(x, lab, Tb, Lb, bl, head, dtype=np.float64)
    assert ok.all() and okc.all()
    for b in range(B):
        gc[Tb[b]:, b] = 0.0                      # the C restatement leaves padded frames to its caller's buffer
    np.testing.assert_allclose(lo, lt, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(lc, lt, rtol=1e-11, atol=1e-11)
    np.testing.assert_allclose(go, gt, rtol=0, atol=2e-8)
    np.testing.assert_allclose(gc, go, rtol=1e-9, atol=1e-11)


def test_param_layer_status_words():
    """param_layer on a hand-written table: truncation toward zero, clamps, which clamps report CTCB_UTT_LEN_CLAMPED (4),
    which labels report CTCB_UTT_BAD_LABEL (2), feasibility on the clamped labels (CTCB_UTT_INFEASIBLE, 1)."""
    T, V = 10, 7
    #            labels (blank 0)              T_b       L_b    -> T_b L_b status
    table = [([1, 2, 3, 4], 10, 4, 10, 4, 0),
             ([1, 2, 3, 4], 10.9, 3.9, 10, 3, 0),         # fractional: truncated, no bit
             ([1, 2, 3, 4], 11, 4, 10, 4, 4),             # > T
             ([1, 2, 3, 4], -1, 4, 0, 4, 4 | 1),          # negative: 0 frames
             ([1, 2, 3, 4], -0.9, 4, 0, 4, 1),            # truncates to 0: no clamp
             ([1, 2, 3, 4], 0, 4, 0, 4, 1),               # no frames
             ([1, 2, 3, 4], 2 ** 40, 4, 10, 4, 4),        # huge
             ([1, 2, 3, 4], 10, 5, 10, 4, 4),             # > Lmax
             ([1, 2, 3, 4], 10, -3, 10, 0, 4),            # negative: empty label sequence
             ([1, 7, 3, 4], 10, 4, 10, 4, 2),             # == V
             ([1, 2, -1, 4], 10, 4, 10, 4, 2),            # negative label
             ([1, 2, 3, -1], 10, 3, 10, 3, 0),            # a bad label past L_b is not read
             ([1, 0, 3, 4], 10, 4, 10, 4, 2),             # == blank
             ([1, 2.9, -0.9, 4], 10, 4, 10, 4, 2),        # -0.9 truncates to 0 == blank; 2.9 -> 2
             ([1e10, 9, 3, 4], 10, 4, 10, 4, 2),          # 1e10 and 9 both clamp to 6: a repeat (5 frames)
             ([1e10, 9, 3, 4], 4, 4, 4, 4, 2 | 1),        # ... so 4 frames are too few
             ([0, 0, 0, 0], 7, 4, 7, 4, 2),               # all blank: 3 repeats, 7 frames suffice
             ([0, 0, 0, 0], 6, 4, 6, 4, 2 | 1),
             ([1, 2, 3, 4], 12.5, 9, 10, 4, 4)]           # both clamped: one bit
    lab = np.array([r[0] for r in table], np.float64)
    dl = np.array([r[1] for r in table], np.float64)
    ll = np.array([r[2] for r in table], np.float64)
    Tb, Lb, labc, st = O.param_layer(lab, dl, ll, T, V, "first")
    assert list(Tb) == [r[3] for r in table]
    assert list(Lb) == [r[4] for r in table]
    assert list(st) == [r[5] for r in table]
    assert labc.min() >= 0 and labc.max() <= V - 1 and labc[13].tolist() == [1, 2, 0, 4]
    # inferred lengths: the first TRUNCATED label equal to the padding value (0 blank first, -1 blank last), unclamped
    lab = np.array([[3, 2, 0, 5], [3, -0.5, 2, 1], [0, 1, 2, 3], [1, 2, 3, 4], [9, -3, 0, 1]], np.float32)
    Tb, Lb, _, st = O.param_layer(lab, None, None, T, V, "first")
    assert list(Tb) == [T] * 5 and list(Lb) == [2, 1, 0, 4, 2] and list(st) == [0, 0, 0, 0, 2]
    lab = np.array([[3, 2, -1, 5], [3, -1.5, 2, 1], [-1, 1, 2, 3], [0, 6, 3, 4], [9, -3, -1, 1]], np.float32)
    _, Lb, labc, st = O.param_layer(lab, None, None, T, V, "last")
    assert list(Lb) == [2, 1, 0, 4, 2] and list(st) == [0, 0, 0, 2, 2]
    assert labc[4, :2].tolist() == [6, 0]
    # integer dtypes give the same answer as the float dtypes holding the same values
    for dt in (np.int32, np.int64):
        _, Lb2, labc2, st2 = O.param_layer(lab.astype(np.float64).astype(dt), None, None, T, V, "last")
        assert list(Lb2) == list(Lb) and list(st2) == list(st) and (labc2 == labc).all()


@pytest.mark.parametrize("blank_last,inferred", [(False, False), (True, False), (False, True), (True, True)])
def test_oracles_agree_on_out_of_range_inputs(blank_last, inferred):
    """The numpy and the C oracle (1e-11) on the hostile batch: labels >= V, negative, fractional, huge, equal to the
    blank; lengths beyond T and Lmax, negative, fractional, huge; inferred label lengths.  Both clamp as the operator
    does; infeasible rows are exactly 0.  The C oracle takes the labels unclamped (it clamps while building the lattice)."""
    from tests.synth import hostile_batch
    T, V, Lmax = 40, 11, 12
    bl = "last" if blank_last else "first"
    for ld, nd in (("f32", "f64"), ("i64", "i32"), ("f64", "i64")):
        d = hostile_batch(T, V, Lmax, blank_last=blank_last, label_dtype=ld, length_dtype=nd, inferred=inferred, seed=3)
        B = d["pred"].shape[0]
        head = np.linspace(0.5, 1.5, B)
        lo, go, ok = O.CtcLossOracle("NTC", "NT", bl)(d["pred"], d["label"], d["pred_lengths"], d["label_lengths"],
                                                      head_grad=head)
        Tb, Lb, labc, st = O.param_layer(d["label"], d["pred_lengths"], d["label_lengths"], T, V, bl)
        np.testing.assert_array_equal(ok, (st & 1) == 0)
        assert (st & 1).any() and (st & 2).any() and ((st & 4).any() or inferred)
        assert (lo[~ok] == 0).all() and (go[~ok] == 0).all() and np.isfinite(lo).all()
        lc, gc, okc = R.ctc_ref(d["pred"], d["label"], Tb, Lb, blank=V - 1 if blank_last else 0, head_grad=head,
                                layout="NTC", dtype=np.float64)
        np.testing.assert_array_equal(okc, ok)
        for b in range(B):
            gc[b, Tb[b]:] = 0.0
        np.testing.assert_allclose(lc, lo, rtol=1e-11, atol=1e-11)
        np.testing.assert_allclose(gc, go, rtol=1e-9, atol=1e-11)
        # the raw lengths straight into the C oracle: it clamps them itself (huge values saturate on the way to int32)
        if not inferred:
            lc2, _, _ = R.ctc_ref(d["pred"], d["label"], d["pred_lengths"], d["label_lengths"],
                                  blank=V - 1 if blank_last else 0, head_grad=head, layout="NTC", dtype=np.float64)
            np.testing.assert_array_equal(lc2, lc)


def test_greedy_decode_clamps_lengths():
    """Frame counts are truncated toward zero and clamped to [0, T]: a negative one decodes nothing (it does not
    slice from the end), one beyond T decodes every frame."""
    rng = np.random.default_rng(4)
    x = rng.standard_normal((5, 12, 6))
    full = O.greedy_decode(x, [12] * 5)
    assert O.greedy_decode(x, np.array([-3, 40, 7.9, -0.5, 2 ** 40], dtype=np.float64)) == [
        [], full[1], O.greedy_decode(x[2:3], [7])[0], [], full[4]]
    assert O.greedy_decode_unk(x, np.array([-3, 40, 5, 0, 12], np.int64), unk=2) == [
        [], O.greedy_decode_unk(x[1:2], [12], 2)[0], O.greedy_decode_unk(x[2:3], [5], 2)[0], [],
        O.greedy_decode_unk(x[4:5], [12], 2)[0]]
