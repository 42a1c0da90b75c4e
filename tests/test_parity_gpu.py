"""GPU parity tests proper: the CUDA path (through the C ABI) against the fp64 oracle, the
committed golden vectors and size-independent properties.  Bar (BASELINE.json north_star):
per-utterance loss and logit gradient within rtol 1e-4 / atol 1e-5 of the oracle."""
import json
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import ctc_oracle as O
from tests.synth import CONFIGS, make_batch

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-4, 1e-5


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _to(dev, d, int_labels=False):
    out = {k: torch.tensor(v, device=dev) for k, v in d.items()}
    if int_labels:
        out["label"] = out["label"].to(torch.int32)
    return out


def _run_block(dev, d, layout="NTC", label_layout="NT", blank_label="first", head=None, lengths=True):
    from gluon_e2e_asr_b200 import CtcLoss
    t = _to(dev, d)
    pred = t["pred"] if layout == "NTC" else t["pred"].transpose(0, 1).contiguous()
    pred.requires_grad_(True)
    lab = t["label"] if label_layout == "NT" else t["label"].t().contiguous()
    blk = CtcLoss(layout=layout, label_layout=label_layout, blank_label=blank_label)
    loss = blk(pred, lab, t["pred_lengths"] if lengths else None, t["label_lengths"] if lengths else None)
    h = torch.ones_like(loss) if head is None else torch.tensor(head, device=dev, dtype=torch.float32)
    (loss * h).sum().backward()
    g = pred.grad
    if layout == "TNC":
        g = g.transpose(0, 1)
    return loss.detach().cpu().numpy(), g.cpu().numpy()


def _oracle(d, blank_label="first", head=None, lengths=True):
    o = O.CtcLossOracle("NTC", "NT", blank_label)
    return o(d["pred"], d["label"], d["pred_lengths"] if lengths else None,
             d["label_lengths"] if lengths else None, head_grad=head)


def _check(loss, grad, lo, go, name=""):
    np.testing.assert_allclose(loss, lo, rtol=RTOL, atol=ATOL, err_msg=name + " loss")
    np.testing.assert_allclose(grad, go, rtol=RTOL, atol=ATOL, err_msg=name + " grad")


def test_kats_through_the_block(dev, golden_dir):
    from gluon_e2e_asr_b200 import CtcLoss
    with open(os.path.join(golden_dir, "kat.json")) as f:
        kats = json.load(f)
    for k in kats:
        data = torch.tensor(np.array(k["data"], np.float32), device=dev)
        lab = torch.tensor(np.array(k["label"], np.float32), device=dev)
        blk = CtcLoss(layout=k["layout"], label_layout="NT", blank_label=k["blank_label"])
        loss = blk(data, lab).cpu().numpy()
        np.testing.assert_allclose(loss, k["expect"], rtol=max(k["rtol"], 2e-6), err_msg=k["name"])
        # int32 labels give the same answer (upstream runs both)
        loss_i = blk(data, lab.to(torch.int32)).cpu().numpy()
        np.testing.assert_array_equal(loss, loss_i)


def test_raw_operator_surface(dev, golden_dir):
    """ctc_loss(data TNC, label, data_lengths, label_lengths, use_*, blank_label) -- loss.py:134-139."""
    from gluon_e2e_asr_b200 import CTCLoss, ctc_loss
    assert CTCLoss is ctc_loss
    d = make_batch(5, 37, 9, 6, seed=11)
    t = _to(dev, d)
    data = t["pred"].transpose(0, 1).contiguous().requires_grad_(True)
    loss = ctc_loss(data, t["label"], t["pred_lengths"], t["label_lengths"], True, True, "first")
    loss.sum().backward()
    lo, go, ok = _oracle(d)
    assert ok.all()
    _check(loss.detach().cpu().numpy(), data.grad.transpose(0, 1).cpu().numpy(), lo, go, "raw op")
    # lengths passed but flags False -> ignored: T frames, labels end at the first 0
    loss2 = ctc_loss(data.detach(), t["label"], t["pred_lengths"], t["label_lengths"]).cpu().numpy()
    lo2, _, _ = _oracle(d, lengths=False)
    np.testing.assert_allclose(loss2, lo2, rtol=RTOL, atol=ATOL)
    with pytest.raises(ValueError):
        ctc_loss(data.detach(), t["label"], None, None, True, False)
    with pytest.raises(RuntimeError):
        ctc_loss(data.detach().cpu(), t["label"].cpu())


def test_torch_fp64_fixtures(dev, golden_dir):
    from gluon_e2e_asr_b200 import ctc_loss_and_grad
    z = np.load(os.path.join(golden_dir, "torch_fp64.npz"))
    for name in sorted({k.split("/")[0] for k in z.files}):
        c = {k.split("/")[1]: z[k] for k in z.files if k.startswith(name + "/")}
        blank_label = "first" if int(c["blank"]) == 0 else "last"
        data = torch.tensor(c["data"], device=dev)                        # TNC
        loss, grad = ctc_loss_and_grad(data, torch.tensor(c["label"], device=dev),
                                       torch.tensor(c["T_b"], device=dev), torch.tensor(c["L_b"], device=dev),
                                       head_grad=torch.tensor(c["head"], device=dev, dtype=torch.float32),
                                       blank_label=blank_label, layout="TNC")
        _check(loss.cpu().numpy(), grad.cpu().numpy(), c["loss"], c["grad"], name)


@pytest.mark.parametrize("cfg,seed,peaky", [("cfg1", 0, False), ("cfg1", 1, True), ("cfg2", 0, False),
                                            ("cfg2", 2, True), ("cfg4", 0, False), ("cfg4", 1, True)])
def test_configs_vs_oracle(dev, cfg, seed, peaky):
    B, T, V, L = CONFIGS[cfg]
    B = min(B, 8)                      # the oracle is a Python loop over T; keep it to seconds
    d = make_batch(B, T, V, L, seed=seed, peaky=peaky)
    head = np.random.default_rng(seed).uniform(0.5, 1.5, B)
    loss, grad = _run_block(dev, d, head=head)
    lo, go, ok = _oracle(d, head=head)
    assert ok.all()
    _check(loss, grad, lo, go, cfg)


def test_cfg3_wide_vocab_vs_oracle(dev):
    B, T, V, L = CONFIGS["cfg3"]
    d = make_batch(3, T, V, L, seed=3)
    loss, grad = _run_block(dev, d)
    lo, go, ok = _oracle(d)
    _check(loss, grad, lo, go, "cfg3")


def test_layouts_and_label_dtypes_agree(dev):
    d = make_batch(6, 50, 13, 10, seed=4)
    base_l, base_g = _run_block(dev, d)
    for layout, ll in (("TNC", "NT"), ("NTC", "TN"), ("TNC", "TN")):
        l, g = _run_block(dev, d, layout=layout, label_layout=ll)
        np.testing.assert_array_equal(l, base_l)
        np.testing.assert_array_equal(g, base_g)
    lo, go, _ = _oracle(d)
    _check(base_l, base_g, lo, go, "layouts")


def test_blank_last_and_inferred_lengths(dev):
    d = make_batch(5, 40, 8, 7, seed=5, blank=7)
    loss, grad = _run_block(dev, d, blank_label="last", lengths=False)
    lo, go, ok = _oracle(d, blank_label="last", lengths=False)
    # without pred_lengths every utterance has T frames: some may become infeasible -> both agree
    _check(loss, grad, lo, go, "blank last")


def test_edge_cases(dev):
    from gluon_e2e_asr_b200 import ctc_loss_and_grad
    rng = np.random.default_rng(9)
    T, B, V, L = 12, 6, 7, 5
    x = rng.standard_normal((B, T, V)).astype(np.float32)
    lab = np.array([[1, 1, 1, 1, 1],      # all repeats: needs 9 frames
                    [1, 2, 3, 4, 5],
                    [0, 0, 0, 0, 0],      # empty label (L=0)
                    [3, 3, 2, 2, 1],      # infeasible with T_b = 6 (needs 7)
                    [6, 5, 4, 3, 2],      # T_b == L_b: single path
                    [2, 2, 0, 0, 0]], np.float32)
    Tb = np.array([9, 12, 7, 6, 5, 3], np.float32)
    Lb = np.array([5, 5, 0, 5, 5, 2], np.float32)
    d = dict(pred=x, label=lab, pred_lengths=Tb, label_lengths=Lb)
    t = _to(dev, d)
    status = torch.zeros((B,), dtype=torch.int32, device=dev)
    loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"], status=status)
    lo, go, ok = _oracle(d)
    assert list(ok) == [True, True, True, False, True, True]
    _check(loss.cpu().numpy(), grad.cpu().numpy(), lo, go, "edge")
    st = status.cpu().numpy()
    assert st[3] & 1 and not (st[[0, 1, 2, 4, 5]] & 1).any()
    assert np.all(grad.cpu().numpy()[3] == 0) and loss[3].item() == 0
    # padded frames are exactly zero
    g = grad.cpu().numpy()
    for b in range(B):
        assert np.all(g[b, int(Tb[b]):] == 0)


def test_properties_at_full_size(dev):
    """cfg2 / cfg5-sized batches without the oracle: row sums, padding zeros, batch == single,
    head-gradient linearity, determinism."""
    from gluon_e2e_asr_b200 import ctc_loss_and_grad
    B, T, V, L = CONFIGS["cfg2"]
    d = make_batch(B, T, V, L, seed=6)
    t = _to(dev, d)
    args = (t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
    loss, grad = ctc_loss_and_grad(*args)
    loss, grad = loss.clone(), grad.clone()
    assert torch.isfinite(loss).all() and torch.isfinite(grad).all()
    Tb = t["pred_lengths"].long()
    mask = torch.arange(T, device=dev)[None, :] < Tb[:, None]
    assert grad[~mask].abs().max().item() == 0
    assert grad.sum(-1)[mask].abs().max().item() < 5e-6          # sum_v G = 0 on valid frames
    # determinism: same bits on a second run
    loss2, grad2 = ctc_loss_and_grad(*args)
    assert torch.equal(loss, loss2) and torch.equal(grad, grad2)
    # linearity in head_grad
    head = torch.linspace(0.5, 2.0, B, device=dev)
    _, gh = ctc_loss_and_grad(*args, head_grad=head)
    torch.testing.assert_close(gh, grad * head[:, None, None], rtol=1e-6, atol=1e-9)
    # batch == single utterance
    for b in (0, B // 2, B - 1):
        l1, g1 = ctc_loss_and_grad(t["pred"][b:b + 1], t["label"][b:b + 1], t["pred_lengths"][b:b + 1],
                                   t["label_lengths"][b:b + 1])
        assert torch.equal(l1[0], loss[b]) and torch.equal(g1[0], grad[b])


def test_autograd_path_equals_fused_path_and_handoffs(dev):
    from gluon_e2e_asr_b200 import CtcLoss, ctc_loss_and_grad
    d = make_batch(7, 80, 46, 20, seed=8)
    t = _to(dev, d)
    blk = CtcLoss()
    pred = t["pred"].clone().requires_grad_(True)
    loss = blk(pred, t["label"], t["pred_lengths"], t["label_lengths"])
    loss.mean().backward()
    head = torch.full((7,), 1.0 / 7, device=dev)
    for handoff in ("dlpack", "pointer"):
        lf, gf = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"], head_grad=head,
                                   handoff=handoff)
        assert torch.equal(lf, loss.detach()) and torch.equal(gf, pred.grad)
    # the two differentiable paths (gradient stored in Forward and scaled in Backward, or history
    # kept and head*G written once in Backward) give the same bits
    from gluon_e2e_asr_b200 import ops
    saved = ops._FUSE_IN_FORWARD_MAX_ELEMS
    try:
        ops._FUSE_IN_FORWARD_MAX_ELEMS = 0
        pred2 = t["pred"].clone().requires_grad_(True)
        loss2 = blk(pred2, t["label"], t["pred_lengths"], t["label_lengths"])
        loss2.mean().backward()
    finally:
        ops._FUSE_IN_FORWARD_MAX_ELEMS = saved
    assert torch.equal(loss2.detach(), loss.detach())
    torch.testing.assert_close(pred2.grad, pred.grad, rtol=2e-7, atol=1e-12)
    # forward-only (evaluation path, train_ctc_ce.py:143): same loss, no history kept
    with torch.no_grad():
        le = blk(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
    assert torch.equal(le, loss.detach())


def test_loss_sum_and_host_entry(dev):
    import ctypes
    from gluon_e2e_asr_b200 import _lib, ctc_loss_and_grad
    d = make_batch(4, 30, 11, 6, seed=10)
    t = _to(dev, d)
    s = torch.zeros((), dtype=torch.float64, device=dev)
    loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"], loss_sum=s)
    assert abs(s.item() - loss.double().sum().item()) < 1e-4
    # host-buffer entry: numpy in, numpy out
    x = np.ascontiguousarray(d["pred"]); g = np.empty_like(x); l = np.empty((4,), np.float32)
    p = _lib.Problem()
    p.T, p.B, p.V, p.Lmax, p.blank, p.label_pad = 30, 4, 11, 6, 0, 0
    p.logits, p.logits_stride_t, p.logits_stride_b = x.ctypes.data, 11, 30 * 11
    p.grad, p.grad_stride_t, p.grad_stride_b = g.ctypes.data, 11, 30 * 11
    lab = np.ascontiguousarray(d["label"]); p.labels, p.label_dtype = lab.ctypes.data, _lib.DT_F32
    p.label_stride_b, p.label_stride_l = 6, 1
    p.data_lengths, p.data_lengths_dtype = d["pred_lengths"].ctypes.data, _lib.DT_F32
    p.label_lengths, p.label_lengths_dtype = d["label_lengths"].ctypes.data, _lib.DT_F32
    p.loss = l.ctypes.data
    _lib.check(_lib.load().ctcb_loss_grad_host(ctypes.byref(p), 0))
    np.testing.assert_array_equal(l, loss.cpu().numpy())
    np.testing.assert_array_equal(g, grad.cpu().numpy())


def test_errors_do_not_fall_back(dev):
    import ctypes
    from gluon_e2e_asr_b200 import _lib
    p = _lib.Problem()
    rc = _lib.load().ctcb_loss_grad(ctypes.byref(p), None, 0, None)
    assert rc == _lib.CTCB_INVALID_VALUE and b"bad shape" in _lib.load().ctcb_last_error()
    x = np.zeros((2, 3, 4), np.float32); l = np.zeros((2,), np.float32)
    p.T, p.B, p.V, p.Lmax = 3, 2, 4, 0
    p.logits, p.loss = x.ctypes.data, l.ctypes.data           # host pointers on the device entry
    ws = torch.empty((1 << 20,), dtype=torch.uint8, device=dev)
    rc = _lib.load().ctcb_loss_grad(ctypes.byref(p), ws.data_ptr(), ws.numel(), None)
    assert rc == _lib.CTCB_INVALID_VALUE
    p.logits = ws.data_ptr(); p.loss = ws.data_ptr() + 4096
    rc = _lib.load().ctcb_loss_grad(ctypes.byref(p), ws.data_ptr() + 8192, 16, None)
    assert rc == _lib.CTCB_WORKSPACE_TOO_SMALL


def test_greedy_decode(dev):
    from gluon_e2e_asr_b200 import greedy_decode
    d = make_batch(6, 70, 46, 15, seed=12, peaky=True)
    t = _to(dev, d)
    toks, lens = greedy_decode(t["pred"], t["pred_lengths"])
    ref = O.greedy_decode(d["pred"], d["pred_lengths"])
    toks, lens = toks.cpu().numpy(), lens.cpu().numpy()
    for b in range(6):
        assert list(toks[b, :lens[b]]) == ref[b]


def test_greedy_decode_unk_rule(dev):
    """decode_ctc.py:120-140: <unk> frames take the second-best symbol, the repeat test compares with the
    RAW best symbol of the previous frame.  Bit-exact against the oracle's loop-for-loop restatement, on
    logits where <unk> wins a third of the frames (runs of <unk>, <unk> next to its substitute, ties)."""
    from gluon_e2e_asr_b200 import greedy_decode
    rng = np.random.default_rng(77)
    B, T, V, unk = 7, 90, 12, 5
    x = rng.standard_normal((B, T, V)).astype(np.float32)
    win = rng.random((B, T)) < 0.35
    x[win, unk] += 6.0                                       # <unk> is the best symbol on these frames
    x[0, 10:20, 3] = 4.0; x[0, 10:20, unk] = 9.0             # a run of <unk> over a constant second best
    x[1, 5, :] = 0.0                                         # an all-ties frame: best 0 (blank), second 1
    x[2, 30:34, unk] = 7.0; x[2, 30:34, 0] = 6.0             # <unk> over blank: substituted symbol is the blank
    lens = np.array([90, 77, 90, 1, 0, 33, 64], np.float32)
    t = torch.tensor(x, device=dev)
    for layout, xt in (("NTC", t), ("TNC", t.transpose(0, 1).contiguous())):
        toks, n = greedy_decode(xt, torch.tensor(lens, device=dev), unk=unk, layout=layout)
        ref = O.greedy_decode_unk(x, lens, unk)
        toks, n = toks.cpu().numpy(), n.cpu().numpy()
        for b in range(B):
            assert list(toks[b, :n[b]]) == ref[b], (layout, b)
    # unk=None is the plain decode
    toks, n = greedy_decode(t, torch.tensor(lens, device=dev))
    ref = O.greedy_decode(x, lens)
    for b in range(B):
        assert list(toks.cpu().numpy()[b, :n.cpu().numpy()[b]]) == ref[b]


def test_wide_logit_ranges_are_floored_and_reported(dev):
    """Emissions are floored at 2^-100 (69.3 nats) below the frame's largest softmax numerator -- a documented
    contract difference (include/ctcb.h CTCB_UTT_WIDE_LOGITS).  Inside that range: parity with the oracle and no
    status bit, up to gaps of 65 nats.  Beyond it: the bit is raised, results stay finite, the loss is the floored
    lattice's (never above the exact one), for the small-vocabulary and the wide-vocabulary path."""
    from gluon_e2e_asr_b200 import _lib, ctc_loss_and_grad
    for V in (46, 300):
        B, T, L = 4, 40, 8
        d = make_batch(B, T, V, L, seed=90 + V)
        rng = np.random.default_rng(V)
        # (a) gaps up to 65 nats: one confident symbol per frame, the rest 55..65 nats below
        x = (rng.uniform(-65.0, -55.0, (B, T, V))).astype(np.float32)
        hot = rng.integers(0, V, (B, T))
        np.put_along_axis(x, hot[..., None], 0.0, axis=2)
        d["pred"] = x
        t = _to(dev, d)
        st = torch.full((B,), -1, dtype=torch.int32, device=dev)
        loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"], status=st)
        lo, go, ok = _oracle(d)
        _check(loss.cpu().numpy(), grad.cpu().numpy(), lo, go, "gaps <= 65 nats, V=%d" % V)
        assert (st.cpu().numpy() & _lib.UTT_WIDE_LOGITS == 0).all()
        # (b) a confident-wrong frame 90 nats above everything the utterance can emit
        y = d["pred"].copy()
        y[:, 7, :] = -90.0
        y[:, 7, V - 1] = 0.0
        for b in range(B):                                     # make sure V-1 is not one of utterance b's labels
            lab = d["label"][b]; lab[lab == V - 1] = 1
        d["pred"] = y
        t = _to(dev, d)
        st = torch.zeros((B,), dtype=torch.int32, device=dev)
        loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"], status=st)
        lo, go, ok = _oracle(d)
        l = loss.cpu().numpy()
        assert np.isfinite(l).all() and torch.isfinite(grad).all()
        assert (st.cpu().numpy() & _lib.UTT_WIDE_LOGITS != 0).all()
        assert (l <= lo + 1e-3).all() and (l >= lo - 25.0).all()          # 90 - 69.3 nats of one frame, at most
        valid = np.arange(T)[None, :] < d["pred_lengths"][:, None]
        rows = grad.cpu().numpy().sum(axis=2)
        assert np.abs(rows[valid]).max() < 1e-4                            # still a gradient of a normalised model


def test_backward_on_a_foreign_workspace_fails_instead_of_hanging(dev):
    """ctcb_backward on a workspace that no matching ctcb_forward filled: the gradient kernel's waits are bounded
    and stamped -- NaN rows come back, the GPU does not hang (ADVICE r1)."""
    import ctypes
    from gluon_e2e_asr_b200 import _lib, ops
    d = make_batch(3, 40, 46, 8, seed=95)
    t = _to(dev, d)
    call = ops._Call(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"], False, True, False)
    ws = torch.zeros((_lib.workspace_bytes(call.T, call.B, call.V, call.Lmax, True),), dtype=torch.uint8, device=dev)
    loss = torch.zeros((3,), device=dev); grad = torch.zeros_like(t["pred"])
    # a forward of ANOTHER shape into the same buffer, then the backward of this one
    d2 = make_batch(3, 32, 46, 8, seed=96)
    t2 = _to(dev, d2)
    call2 = ops._Call(t2["pred"], t2["label"], t2["pred_lengths"], t2["label_lengths"], False, True, False)
    call2.run(_lib.PHASE_FORWARD, ws, loss, keep=True, handoff="pointer")
    call.run(_lib.PHASE_BACKWARD, ws, loss, grad=grad, handoff="pointer")
    torch.cuda.synchronize()
    assert torch.isnan(grad).all()
    # the matching pair still works afterwards
    call.run(_lib.PHASE_FORWARD, ws, loss, keep=True, handoff="pointer")
    call.run(_lib.PHASE_BACKWARD, ws, loss, grad=grad, handoff="pointer")
    lo, go, _ = _oracle(d)
    _check(loss.cpu().numpy(), grad.cpu().numpy(), lo, go, "forward + backward")


def _env(**kw):
    """Context manager: set libctcb's tuning switches (ctcb_set_option; CTCB_OVERLAP=0 -> option "overlap")."""
    from gluon_e2e_asr_b200 import _lib
    return _lib.options(**{k[5:].lower() if k.startswith("CTCB_") else k: v for k, v in kw.items()})


def test_overlapped_and_serial_schedules_agree(dev):
    """k_grad as a programmatic dependent of k_walk (progress flags, SM partitioning) against the
    kernels launched one after the other.  The overlapped schedule gives the same BITS run after
    run (a race between the walkers and the gradient CTAs would show) and under a different SM
    partition; the serial schedule launches the high-occupancy build of the same gradient kernel,
    whose floating-point contractions may differ in the last bit, so it is compared to 1e-6."""
    from gluon_e2e_asr_b200 import ctc_loss_and_grad, ops
    B, T, V, L = CONFIGS["cfg2"]
    d = make_batch(B, T, V, L, seed=21)
    t = _to(dev, d)
    args = (t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
    with _env(CTCB_OVERLAP=0):
        ops._ws_cache.clear()
        l0, g0 = ctc_loss_and_grad(*args)
        l0, g0 = l0.clone(), g0.clone()
    ref = None
    for rep in range(5):
        with _env(CTCB_OVERLAP=1):
            l1, g1 = ctc_loss_and_grad(*args, out_grad=torch.full_like(g0, float("nan")))
        if ref is None:
            ref = (l1.clone(), g1.clone())
        assert torch.equal(ref[0], l1) and torch.equal(ref[1], g1), "overlap run %d differs" % rep
    assert torch.equal(l0, ref[0])
    torch.testing.assert_close(ref[1], g0, rtol=1e-6, atol=1e-7)
    with _env(CTCB_OVERLAP=1, CTCB_WALK_PER_SM=2):
        l2, g2 = ctc_loss_and_grad(*args)
    assert torch.equal(ref[0], l2) and torch.equal(ref[1], g2)


def test_wide_vocabulary_schedules_agree(dev):
    """Wide vocabularies (rows staged by bulk copies): k_emit, then k_walk with k_grad as its programmatic
    dependent sharing the walkers' SMs, against the same kernels launched one after the other: same BITS
    (loss, gradient, status), run after run, for ragged batches with an infeasible utterance; and inside
    the tolerance of the fp64 oracle."""
    from gluon_e2e_asr_b200 import ctc_loss_and_grad, ops
    for (B, T, V, L, seed) in ((9, 75, 600, 14, 41), (5, 130, 2000, 40, 42), (64, 40, 1024, 9, 43)):
        d = make_batch(B, T, V, L, seed=seed)
        d["pred_lengths"][1] = 4.0; d["label_lengths"][1] = float(min(L, 9))       # infeasible
        t = _to(dev, d)
        args = (t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
        head = torch.linspace(0.5, 1.5, B, device=dev)
        with _env(CTCB_OVERLAP=0):
            ops._ws_cache.clear()
            st0 = torch.zeros((B,), dtype=torch.int32, device=dev)
            l0, g0 = ctc_loss_and_grad(*args, head_grad=head, status=st0)
            l0, g0 = l0.clone(), g0.clone()
            assert _lib_launches() == 3
        for rep in range(4):
            st1 = torch.zeros((B,), dtype=torch.int32, device=dev)
            with _env(CTCB_OVERLAP=1):
                l1, g1 = ctc_loss_and_grad(*args, head_grad=head, status=st1, out_grad=torch.full_like(g0, float("nan")))
            assert _lib_launches() == 3
            assert torch.equal(l0, l1) and torch.equal(st0, st1), "loss/status differ (run %d)" % rep
            assert torch.equal(g0, g1), "gradient differs (run %d)" % rep
        lo, go, ok = O.CtcLossOracle("NTC", "NT")(d["pred"], d["label"], d["pred_lengths"], d["label_lengths"],
                                                 head_grad=head.cpu().numpy().astype(np.float64))
        _check(l1.cpu().numpy(), g1.cpu().numpy(), lo, go, "wide overlapped B%d T%d V%d" % (B, T, V))
        assert (st1.cpu().numpy()[1] & 1) == 1 and not ok[1]


def _lib_launches():
    from gluon_e2e_asr_b200 import _lib
    return _lib.last_launch_count()


def test_fused_and_unfused_emissions_agree(dev):
    """Emission blocks made by the walkers' producer warps (V <= 64) against k_emit + TMA: the same
    numerators; only the summation order of the loss normaliser differs."""
    from gluon_e2e_asr_b200 import ctc_loss_and_grad, ops
    d = make_batch(8, 200, 46, 50, seed=22)
    t = _to(dev, d)
    args = (t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
    lf, gf = ctc_loss_and_grad(*args)
    lf, gf = lf.clone(), gf.clone()
    with _env(CTCB_FUSED=0):
        ops._ws_cache.clear()                      # the workspace layout differs (emission table)
        lu, gu = ctc_loss_and_grad(*args)
    ops._ws_cache.clear()
    torch.testing.assert_close(lf, lu, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(gf, gu, rtol=1e-5, atol=1e-7)
    # odd vocabulary / TNC strides / blank last go through the fused producers too
    d = make_batch(5, 61, 63, 9, seed=23, blank=62)
    loss, grad = _run_block(dev, d, layout="TNC", blank_label="last")
    lo, go, _ = _oracle(d, blank_label="last")
    _check(loss, grad, lo, go, "fused V=63 TNC blank last")


def test_step_replays_from_a_cuda_graph(dev):
    """The two-kernel step (programmatic dependency included) captured once and replayed."""
    from gluon_e2e_asr_b200 import ctc_loss_and_grad
    d = make_batch(16, 120, 46, 30, seed=24)
    t = _to(dev, d)
    args = (t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
    l0, g0 = ctc_loss_and_grad(*args)
    l0, g0 = l0.clone(), g0.clone()
    loss = torch.empty_like(l0); grad = torch.empty_like(g0)
    s = torch.cuda.Stream(dev)
    with torch.cuda.stream(s):
        ctc_loss_and_grad(*args, out_loss=loss, out_grad=grad, handoff="pointer")      # warm the workspace cache
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            ctc_loss_and_grad(*args, out_loss=loss, out_grad=grad, handoff="pointer")
        for _ in range(3):
            loss.fill_(float("nan")); grad.fill_(float("nan"))
            g.replay()
            torch.cuda.synchronize()
            assert torch.equal(loss, l0) and torch.equal(grad, g0)


def test_batch_larger_than_the_resident_walkers(dev):
    """B > 296: the walkers do not fit the GPU at once, k_grad is a plain launch after them."""
    from gluon_e2e_asr_b200 import ctc_loss_and_grad
    d = make_batch(320, 24, 11, 6, seed=25)
    t = _to(dev, d)
    loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
    lo, go, _ = _oracle(d)
    _check(loss.cpu().numpy(), grad.cpu().numpy(), lo, go, "B=320")


def test_pinned_batch_single_copy(dev):
    from gluon_e2e_asr_b200 import CtcLoss
    from gluon_e2e_asr_b200.batch import PinnedBatch
    d = make_batch(4, 60, 46, 12, seed=26)
    pb = PinnedBatch.from_arrays(d["pred"], d["label"], d["pred_lengths"], d["label_lengths"])
    assert pb.arena.is_pinned()
    x = pb.load(dev)
    assert x["pred"].data_ptr() % 256 == 0 and x["label"].data_ptr() % 256 == 0
    pred = x["pred"].requires_grad_(True)
    loss = CtcLoss()(pred, x["label"], x["pred_lengths"], x["label_lengths"])
    loss.sum().backward()
    lo, go, _ = _oracle(d)
    _check(loss.detach().cpu().numpy(), pred.grad.cpu().numpy(), lo, go, "pinned batch")
    assert pb.load(dev)["pred"] is x["pred"]                    # persistent device arena, same views


@pytest.mark.parametrize("B,T,V,L,seed", [
    (2, 2300, 30, 2047, 40),      # the longest label row the library takes: 16 walker warps x 4 pairs per lane
    (2, 1500, 30, 700, 41),       # 12 walker warps
    (3, 900, 64, 200, 42),        # widest fused vocabulary
    (3, 300, 65, 40, 43),         # narrowest unfused vocabulary (k_emit + TMA, dense table)
    (4, 64, 2, 20, 44),           # V = 2: blank and one symbol, every neighbour a repeat
    (1, 1, 5, 1, 45),             # one frame, one label
])
def test_extreme_shapes_vs_oracle(dev, B, T, V, L, seed):
    d = make_batch(B, T, V, L, seed=seed)
    loss, grad = _run_block(dev, d)
    lo, go, ok = _oracle(d)
    _check(loss, grad, lo, go, "B%d T%d V%d L%d" % (B, T, V, L))


def test_strided_views_and_wide_logit_range(dev):
    """Logits that are a slice of a larger tensor (T and B strides not compact, V stride 1), and a
    logit spread of +-30 (per-frame probabilities down to e^-60)."""
    from gluon_e2e_asr_b200 import ctc_loss_and_grad
    d = make_batch(5, 90, 46, 20, seed=46, scale=12.0)
    big = torch.zeros((7, 100, 46 + 18), device=dev)
    big[1:6, 4:94, 9:55] = torch.tensor(d["pred"], device=dev)
    view = big[1:6, 4:94, 9:55]
    assert not view.is_contiguous() and view.stride(2) == 1
    t = _to(dev, d)
    out = torch.zeros_like(big)
    gview = out[1:6, 4:94, 9:55]
    loss, grad = ctc_loss_and_grad(view, t["label"], t["pred_lengths"], t["label_lengths"], out_grad=gview)
    lo, go, ok = _oracle(d)
    assert ok.all()
    _check(loss.cpu().numpy(), gview.cpu().numpy(), lo, go, "strided")
    assert out[0].abs().max().item() == 0 and out[:, :4].abs().max().item() == 0      # nothing written outside the view


def test_host_entry_with_resident_gradient(dev):
    """ctcb_loss_grad_host_resident: host buffers in, loss back, gradient left on the device."""
    import ctypes
    from gluon_e2e_asr_b200 import _lib, ctc_loss_and_grad
    d = make_batch(4, 50, 46, 9, seed=27)
    t = _to(dev, d)
    loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
    x = np.ascontiguousarray(d["pred"]); l = np.empty((4,), np.float32)
    lab = np.ascontiguousarray(d["label"])
    p = _lib.Problem()
    p.T, p.B, p.V, p.Lmax, p.blank, p.label_pad = 50, 4, 46, 9, 0, 0
    p.logits, p.logits_stride_t, p.logits_stride_b = x.ctypes.data, 46, 50 * 46
    p.labels, p.label_dtype, p.label_stride_b, p.label_stride_l = lab.ctypes.data, _lib.DT_F32, 9, 1
    p.data_lengths, p.data_lengths_dtype = d["pred_lengths"].ctypes.data, _lib.DT_F32
    p.label_lengths, p.label_lengths_dtype = d["label_lengths"].ctypes.data, _lib.DT_F32
    p.loss = l.ctypes.data
    dg = ctypes.c_void_p()
    _lib.check(_lib.load().ctcb_loss_grad_host_resident(ctypes.byref(p), 0, ctypes.byref(dg)))
    np.testing.assert_array_equal(l, loss.cpu().numpy())
    got = torch.empty_like(grad)
    assert dg.value
    ctypes.CDLL("libcudart.so.12").cudaMemcpy(ctypes.c_void_p(got.data_ptr()), dg, ctypes.c_size_t(got.numel() * 4), 3)
    assert torch.equal(got, grad)
    assert _lib.load().ctcb_loss_grad_host_resident(ctypes.byref(p), 0, None) == _lib.CTCB_INVALID_VALUE


def test_host_entry_full_outputs(dev):
    """ctcb_loss_grad_host with every output (gradient, status, loss sum back on the host, head gradient,
    an infeasible utterance): the same bits as one device call."""
    import ctypes
    from gluon_e2e_asr_b200 import _lib, ctc_loss_and_grad
    B, T, V, L = 19, 70, 46, 14
    d = make_batch(B, T, V, L, seed=28)
    d["pred_lengths"][3] = 5.0; d["label_lengths"][3] = 9.0           # one infeasible utterance
    t = _to(dev, d)
    head = np.linspace(0.5, 1.5, B).astype(np.float32)
    s_dev = torch.zeros((), dtype=torch.float64, device=dev)
    st_dev = torch.zeros((B,), dtype=torch.int32, device=dev)
    loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"],
                                   head_grad=torch.tensor(head, device=dev), loss_sum=s_dev, status=st_dev)
    x = np.ascontiguousarray(d["pred"]); g = np.empty_like(x); l = np.empty((B,), np.float32)
    lab = np.ascontiguousarray(d["label"]); st = np.zeros((B,), np.int32); ssum = np.zeros((1,), np.float64)
    p = _lib.Problem()
    p.T, p.B, p.V, p.Lmax, p.blank, p.label_pad = T, B, V, L, 0, 0
    p.logits, p.logits_stride_t, p.logits_stride_b = x.ctypes.data, V, T * V
    p.grad, p.grad_stride_t, p.grad_stride_b = g.ctypes.data, V, T * V
    p.labels, p.label_dtype, p.label_stride_b, p.label_stride_l = lab.ctypes.data, _lib.DT_F32, L, 1
    p.data_lengths, p.data_lengths_dtype = d["pred_lengths"].ctypes.data, _lib.DT_F32
    p.label_lengths, p.label_lengths_dtype = d["label_lengths"].ctypes.data, _lib.DT_F32
    p.head_grad, p.loss, p.status, p.loss_sum = head.ctypes.data, l.ctypes.data, st.ctypes.data, ssum.ctypes.data
    for rep in range(2):
        g[:] = np.nan; l[:] = np.nan; st[:] = 0; ssum[0] = 0.0
        _lib.check(_lib.load().ctcb_loss_grad_host(ctypes.byref(p), 0))
        np.testing.assert_array_equal(l, loss.cpu().numpy())
        np.testing.assert_array_equal(g, grad.cpu().numpy())
        np.testing.assert_array_equal(st, st_dev.cpu().numpy())
        assert st[3] & 1 and l[3] == 0
        assert abs(ssum[0] - s_dev.item()) < 1e-9 * max(1.0, abs(s_dev.item()))


def test_prefetching_pipe_matches_device_calls(dev):
    """ctcb_pipe_*: batches of changing shape submitted back to back with `depth` in flight; every
    ticket's loss (host) and gradient (device slot) carry the same bits as a plain device call, from
    one-arena pinned batches (one copy) and from separately allocated pageable arrays (one copy per
    array) alike; ticket misuse is an error."""
    import ctypes
    from gluon_e2e_asr_b200 import HostPipeline, PinnedBatch, _lib, ctc_loss_and_grad
    shapes = [(6, 40, 46, 8), (6, 40, 46, 8), (3, 90, 46, 20), (9, 33, 80, 7), (6, 40, 46, 8), (2, 120, 5, 30), (6, 40, 46, 8)]
    for depth in (1, 2, 3):
        pipe = HostPipeline(0, depth=depth)
        want, tickets, keep = [], [], []
        for i, (B, T, V, L) in enumerate(shapes):
            d = make_batch(B, T, V, L, seed=300 + i)
            t = _to(dev, d)
            want.append(ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"]))
            pb = PinnedBatch.from_arrays(d["pred"], d["label"], d["pred_lengths"], d["label_lengths"])
            lo = torch.full((B,), float("nan")).pin_memory()
            keep.append((pb, lo))
            tickets.append(pipe.submit(pb, lo))
            if i >= depth - 1:                                   # collect the oldest batch in flight
                j = i - (depth - 1)
                g = pipe.wait(tickets[j])
                assert torch.equal(keep[j][1], want[j][0].cpu()), (depth, j)
                assert torch.equal(g, want[j][1]), (depth, j)
        for j in range(len(shapes) - (depth - 1), len(shapes)):
            g = pipe.wait(tickets[j])
            assert torch.equal(keep[j][1], want[j][0].cpu()) and torch.equal(g, want[j][1])
        l = _lib.load()
        assert l.ctcb_pipe_wait(pipe._h, 99, None) == _lib.CTCB_INVALID_VALUE
        if depth < len(shapes):
            assert l.ctcb_pipe_wait(pipe._h, 0, None) == _lib.CTCB_INVALID_VALUE      # slot long reused
        pipe.close()
    # one-arena pinned batch whose padded frames are NaN on the host: ONE copy of the arena, and nothing reads the padding
    B, T, V, L = 8, 64, 46, 9
    d = make_batch(B, T, V, L, seed=320)
    d["pred_lengths"][:] = np.array([64, 40, 33, 64, 21, 50, 12, 64], np.float32)
    d["label_lengths"][:] = np.minimum(d["label_lengths"], 5)
    for b in range(B):
        d["pred"][b, int(d["pred_lengths"][b]):] = np.nan
    t = _to(dev, d)
    want = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
    pb = PinnedBatch.from_arrays(d["pred"], d["label"], d["pred_lengths"], d["label_lengths"])
    pipe = HostPipeline(0, depth=2)
    lo = torch.full((B,), float("nan")).pin_memory()
    g = pipe.wait(pipe.submit(pb, lo))
    moved, pulled = pipe.last_h2d_bytes()
    assert not pulled and pb.nbytes - 256 < moved <= pb.nbytes          # one copy of the arena (its last field is not padded)
    assert torch.equal(lo, want[0].cpu()) and torch.equal(g, want[1])
    assert not torch.isnan(g).any()
    pipe.close()
    # PACKED arena (ctcb_problem_t.logits_row_offsets): only the valid frames exist on the host and cross PCIe; same bits
    pk = PinnedBatch.from_arrays(d["pred"], d["label"], d["pred_lengths"], d["label_lengths"], packed=True)
    assert pk.packed and pk.pred.shape == (int(d["pred_lengths"].sum()), V) and not torch.isnan(pk.pred).any()
    pipe = HostPipeline(0, depth=2)
    for rep in range(3):
        lo = torch.full((B,), float("nan")).pin_memory()
        g = pipe.wait(pipe.submit(pk, lo))
        moved, _ = pipe.last_h2d_bytes()
        assert moved <= pk.nbytes and moved < 0.75 * pb.nbytes
        assert torch.equal(lo, want[0].cpu()) and torch.equal(g, want[1])
    pipe.close()
    # the synchronous host entry takes the packed layout too
    q = HostPipeline.problem(None, pk, lo)
    dgp = ctypes.c_void_p()
    lo.fill_(float("nan"))
    _lib.check(_lib.load().ctcb_loss_grad_host_resident(ctypes.byref(q), 0, ctypes.byref(dgp)))
    assert torch.equal(lo, want[0].cpu())
    # separately pinned arrays that are NOT one allocation are never merged into one copy, whatever their addresses
    parts = [torch.tensor(d[k]).pin_memory() for k in ("pred", "label", "pred_lengths", "label_lengths")]
    q = _lib.Problem()
    q.T, q.B, q.V, q.Lmax, q.blank, q.label_pad = T, B, V, L, 0, 0
    q.logits, q.logits_stride_t, q.logits_stride_b = parts[0].data_ptr(), V, T * V
    q.labels, q.label_dtype, q.label_stride_b, q.label_stride_l = parts[1].data_ptr(), _lib.DT_F32, L, 1
    q.data_lengths, q.data_lengths_dtype = parts[2].data_ptr(), _lib.DT_F32
    q.label_lengths, q.label_lengths_dtype = parts[3].data_ptr(), _lib.DT_F32
    lo2 = torch.full((B,), float("nan")).pin_memory()
    q.loss = lo2.data_ptr()
    h = ctypes.c_void_p(); tk = ctypes.c_int64(-1); hb = ctypes.c_int64(0)
    l = _lib.load()
    _lib.check(l.ctcb_pipe_create(0, 2, ctypes.byref(h)))
    _lib.check(l.ctcb_pipe_submit(h, ctypes.byref(q), ctypes.byref(tk)))
    _lib.check(l.ctcb_pipe_wait(h, tk, None))
    _lib.check(l.ctcb_pipe_last_h2d_bytes(h, ctypes.byref(hb), None))
    assert hb.value == sum(x.numel() * 4 for x in parts)               # the arrays' own bytes: no span copy
    assert torch.equal(lo2, want[0].cpu())
    assert l.ctcb_pipe_destroy(h) == _lib.CTCB_OK
    # separately allocated pageable arrays, head gradient, loss sum and status through the raw ABI
    B, T, V, L = 7, 44, 46, 10
    d = make_batch(B, T, V, L, seed=311)
    d["pred_lengths"][2] = 3.0; d["label_lengths"][2] = 8.0          # infeasible
    t = _to(dev, d)
    head = np.linspace(0.5, 1.5, B).astype(np.float32)
    s_dev = torch.zeros((), dtype=torch.float64, device=dev)
    st_dev = torch.zeros((B,), dtype=torch.int32, device=dev)
    loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"],
                                   head_grad=torch.tensor(head, device=dev), loss_sum=s_dev, status=st_dev)
    x = np.ascontiguousarray(d["pred"].transpose(1, 0, 2))           # TNC this time
    lab = np.ascontiguousarray(d["label"]); lh = np.empty((B,), np.float32)
    st = np.zeros((B,), np.int32); ssum = np.zeros((1,), np.float64)
    p = _lib.Problem()
    p.T, p.B, p.V, p.Lmax, p.blank, p.label_pad = T, B, V, L, 0, 0
    p.logits, p.logits_stride_t, p.logits_stride_b = x.ctypes.data, B * V, V
    p.labels, p.label_dtype, p.label_stride_b, p.label_stride_l = lab.ctypes.data, _lib.DT_F32, L, 1
    p.data_lengths, p.data_lengths_dtype = d["pred_lengths"].ctypes.data, _lib.DT_F32
    p.label_lengths, p.label_lengths_dtype = d["label_lengths"].ctypes.data, _lib.DT_F32
    p.head_grad, p.loss, p.status, p.loss_sum = head.ctypes.data, lh.ctypes.data, st.ctypes.data, ssum.ctypes.data
    h = ctypes.c_void_p(); tk = ctypes.c_int64(-1); dg = ctypes.c_void_p()
    l = _lib.load()
    _lib.check(l.ctcb_pipe_create(0, 2, ctypes.byref(h)))
    _lib.check(l.ctcb_pipe_submit(h, ctypes.byref(p), ctypes.byref(tk)))
    _lib.check(l.ctcb_pipe_wait(h, tk, ctypes.byref(dg)))
    got = torch.empty((T, B, V), device=dev)
    ctypes.CDLL("libcudart.so.12").cudaMemcpy(ctypes.c_void_p(got.data_ptr()), dg, ctypes.c_size_t(got.numel() * 4), 3)
    np.testing.assert_array_equal(lh, loss.cpu().numpy())
    assert torch.equal(got.transpose(0, 1), grad)
    np.testing.assert_array_equal(st, st_dev.cpu().numpy())
    assert st[2] & 1 and lh[2] == 0
    assert abs(ssum[0] - s_dev.item()) < 1e-9 * max(1.0, abs(s_dev.item()))
    p.logits_stride_t = 3
    assert l.ctcb_pipe_submit(h, ctypes.byref(p), ctypes.byref(tk)) == _lib.CTCB_INVALID_VALUE
    assert l.ctcb_pipe_destroy(h) == _lib.CTCB_OK


def test_random_small_problems_vs_oracle(dev):
    """Property test (hypothesis): random shapes, vocabularies on both sides of the fused limit, ragged
    and infeasible lengths, both blank conventions, both layouts, int or float labels -- loss, gradient
    and status bits against the fp64 oracle."""
    hyp = pytest.importorskip("hypothesis")
    st = hyp.strategies
    from gluon_e2e_asr_b200 import ctc_loss_and_grad

    @hyp.settings(max_examples=60, deadline=None, derandomize=True,
                  suppress_health_check=list(hyp.HealthCheck))
    @hyp.given(B=st.integers(1, 5), T=st.integers(1, 40), V=st.sampled_from([2, 3, 7, 46, 63, 64, 65, 90]),
               L=st.integers(0, 12), seed=st.integers(0, 10 ** 6), blank_last=st.booleans(), tnc=st.booleans(),
               int_labels=st.booleans(), scale=st.sampled_from([0.3, 1.0, 6.0]))
    def run(B, T, V, L, seed, blank_last, tnc, int_labels, scale):
        rng = np.random.default_rng(seed)
        blank = V - 1 if blank_last else 0
        lo, hi = (0, V - 1) if blank_last else (1, V)
        lab = rng.integers(lo, hi, (B, max(L, 1))).astype(np.float32)
        Lb = rng.integers(0, L + 1, B).astype(np.float32)
        Tb = rng.integers(1, T + 1, B).astype(np.float32)           # some utterances end up infeasible
        x = (rng.standard_normal((B, T, V)) * scale).astype(np.float32)
        head = rng.uniform(0.5, 1.5, B)
        d = dict(pred=x, label=lab, pred_lengths=Tb, label_lengths=Lb)
        o = O.CtcLossOracle("NTC", "NT", "last" if blank_last else "first")
        lo_, go_, ok = o(x, lab, Tb, Lb, head_grad=head)
        xt = torch.tensor(x, device=dev)
        if tnc:
            xt = xt.transpose(0, 1).contiguous()
        labt = torch.tensor(lab, device=dev)
        if int_labels:
            labt = labt.to(torch.int64)
        status = torch.zeros((B,), dtype=torch.int32, device=dev)
        loss, grad = ctc_loss_and_grad(xt, labt, torch.tensor(Tb, device=dev), torch.tensor(Lb, device=dev),
                                       head_grad=torch.tensor(head, device=dev, dtype=torch.float32),
                                       blank_label="last" if blank_last else "first",
                                       layout="TNC" if tnc else "NTC", status=status)
        g = grad.transpose(0, 1) if tnc else grad
        _check(loss.cpu().numpy(), g.cpu().numpy(), lo_, go_, "B%d T%d V%d L%d seed%d" % (B, T, V, L, seed))
        np.testing.assert_array_equal((status.cpu().numpy() & 1) == 0, ok)

    run()


# ---- BASELINE.json configs at their REAL batch sizes ------------------------------------------------
# The numpy oracle is a Python loop over T; at full batch sizes the checker is the oracle's C
# restatement in fp64 (oracle/ctc_ref.c), itself pinned to the numpy oracle at 1e-11 on the golden
# fixtures (tests/test_oracle.py::test_torch_fp64_fixtures_numpy_and_c, test_c_fp64_matches_numpy_at_size).
def _c_oracle(d, head=None):
    from oracle import ctc_ref
    lo, go, ok = ctc_ref.ctc_ref(d["pred"], d["label"], d["pred_lengths"], d["label_lengths"], blank=0,
                                 head_grad=head, layout="NTC", dtype=np.float64)
    return lo, go, ok


@pytest.mark.parametrize("cfg,seed,peaky,full", [
    ("cfg2", 0, False, False), ("cfg2", 1, True, False),
    ("cfg3", 0, False, False),
    ("cfg4", 0, False, False), ("cfg4", 1, True, False),
    ("cfg5", 0, False, False), ("cfg5", 1, False, True), ("cfg5", 2, True, False),
])
def test_baseline_configs_at_full_batch_size(dev, cfg, seed, peaky, full):
    """Loss and gradient at rtol 1e-4 / atol 1e-5 for the BASELINE shapes at their real B (cfg2 32,
    cfg3 64, cfg4 16, cfg5 1024), through ctc_loss_and_grad AND CtcLoss(...).mean().backward()
    (train_ctc_ce.py:363-366)."""
    from gluon_e2e_asr_b200 import CtcLoss, ctc_loss_and_grad
    B, T, V, L = CONFIGS[cfg]
    d = make_batch(B, T, V, L, seed=seed, peaky=peaky, full_lengths=full)
    head = np.full((B,), 1.0 / B)
    lo, go, ok = _c_oracle(d, head=head)
    assert ok.all()
    t = _to(dev, d)
    loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"],
                                   head_grad=torch.tensor(head, device=dev, dtype=torch.float32))
    _check(loss.cpu().numpy(), grad.cpu().numpy(), lo, go, cfg + " fused")
    del grad
    pred = t["pred"].requires_grad_(True)
    l2 = CtcLoss(layout="NTC", label_layout="NT")(pred, t["label"], t["pred_lengths"], t["label_lengths"])
    l2.mean().backward()
    _check(l2.detach().cpu().numpy(), pred.grad.cpu().numpy(), lo, go, cfg + " block.mean().backward()")


@pytest.mark.parametrize("B,T,V,L,seed", [
    (300, 120, 46, 120, 60),     # B > 296 AND L > 32: the plain-launch, register-capped gradient kernel of cfg5
    (100, 200, 46, 50, 61),      # 75 <= B <= 148: two walker CTAs per SM in the shared-memory partition
    (150, 96, 30, 20, 62),       # 149..296: the walkers still fit the GPU at once
])
def test_batch_size_regimes_vs_c_oracle(dev, B, T, V, L, seed):
    from gluon_e2e_asr_b200 import ctc_loss_and_grad
    d = make_batch(B, T, V, L, seed=seed)
    lo, go, ok = _c_oracle(d)
    t = _to(dev, d)
    loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
    _check(loss.cpu().numpy(), grad.cpu().numpy(), lo, go, "B=%d" % B)


# ---- the one-kernel path (ctcb_meet.cuh), opt-in through the "meet" option -----------------------------
@pytest.mark.parametrize("B,T,V,L,seed,peaky", [
    (2, 12, 5, 3, 1, False),        # one frame block more than the labels need
    (3, 7, 46, 2, 3, False),        # a single (partial) frame block: the beta walker has no phase 1
    (3, 9, 46, 4, 4, False),        # two frame blocks
    (5, 100, 33, 40, 5, False),     # P = 2 state pairs per lane
    (6, 64, 64, 31, 6, False),      # P = 1, the widest vocabulary of the path
    (8, 200, 46, 50, 1, True),      # cfg1, peaky
    (32, 500, 46, 120, 0, False),   # cfg2
    (300, 120, 46, 120, 60, False), # more utterances than two per SM
])
def test_meet_in_the_middle_kernel_vs_c_oracle(dev, B, T, V, L, seed, peaky):
    """k_meet (alpha and beta walkers of an utterance meet in the middle, occupancies normalised by P(l|x), one
    launch): same tolerance against the fp64 C oracle as the two-kernel path, head gradients included, and the
    same bits run after run."""
    from gluon_e2e_asr_b200 import ctc_loss_and_grad, ops
    d = make_batch(B, T, V, L, seed=seed, peaky=peaky)
    head = np.linspace(0.5, 2.0, B)
    lo, go, ok = _c_oracle(d, head=head)
    t = _to(dev, d)
    h = torch.tensor(head, device=dev, dtype=torch.float32)
    with _env(meet=1):
        ops._ws_cache.clear()
        loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"], head_grad=h)
        assert _lib_launches() == 1
        l1, g1 = loss.clone(), grad.clone()
        loss2, grad2 = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"], head_grad=h,
                                         out_grad=torch.full_like(grad, float("nan")))
        assert torch.equal(l1, loss2) and torch.equal(g1, grad2)
    ops._ws_cache.clear()
    _check(l1.cpu().numpy(), g1.cpu().numpy(), lo, go, "k_meet B=%d" % B)


def test_meet_kernel_edge_cases(dev):
    """Infeasible utterances (loss 0, gradient 0, status bit), empty labels and a zero-length utterance through k_meet."""
    from gluon_e2e_asr_b200 import ctc_loss_and_grad, ops
    d = make_batch(6, 40, 11, 6, seed=9)
    d["label"][1, :3] = 4; d["label_lengths"][1] = 3; d["pred_lengths"][1] = 4      # 3 repeats need 5 frames: infeasible
    d["label_lengths"][2] = 0                                                         # empty label sequence
    d["pred_lengths"][3] = 0                                                          # no frames at all
    lo, go, ok = _c_oracle(d)
    t = _to(dev, d)
    status = torch.zeros((6,), dtype=torch.int32, device=dev)
    with _env(meet=1):
        ops._ws_cache.clear()
        loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"], status=status)
    ops._ws_cache.clear()
    st = status.cpu().numpy()
    assert st[1] & 1 and st[3] & 1 and not (st[0] & 1) and not (st[2] & 1)
    l, g = loss.cpu().numpy(), grad.cpu().numpy()
    assert l[1] == 0 and l[3] == 0 and not g[1].any() and not g[3].any()
    feas = [0, 2, 4, 5]
    _check(l[feas], g[feas], lo[feas], go[feas], "k_meet edge cases")
    # tight utterances (T_b = L_b + repeats for nine of the 64 rows): beta' is exactly 0 on most states of their late
    # frames, where k_meet must count a state as empty rather than multiply its shifted alpha by zero
    d = make_batch(64, 140, 46, 120, seed=3)
    lo, go, ok = _c_oracle(d)
    assert ok.all()
    t = _to(dev, d)
    with _env(meet=1):
        ops._ws_cache.clear()
        loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
        assert _lib_launches() == 1
    ops._ws_cache.clear()
    assert torch.isfinite(grad).all()
    _check(loss.cpu().numpy(), grad.cpu().numpy(), lo, go, "k_meet tight utterances")


# ---- k_grad2: the gradient kernel that normalises by P(l|x) (ctcb_grad2.cuh) ---------------------------
@pytest.mark.parametrize("B,T,V,L,seed,peaky,blocks", [
    (2, 12, 5, 3, 1, False, 1), (3, 7, 46, 2, 3, False, 4), (5, 100, 33, 40, 5, False, 2), (6, 64, 64, 31, 6, False, 4),
    (8, 200, 46, 50, 1, True, 3), (32, 500, 46, 120, 0, False, 4), (8, 300, 46, 200, 7, False, 2),
    (16, 2000, 46, 300, 0, False, 16), (300, 120, 46, 120, 60, False, 4),
    (4, 1100, 46, 383, 13, False, 2), (3, 1100, 64, 511, 17, False, 4),    # walker configurations (2,6) and (2,8)
    # T barely above L: most utterances have T_b = L_b + repeats, so beta' is exactly 0 on most states of their late frames
    (16, 530, 64, 511, 19, False, 4), (64, 140, 46, 120, 23, False, 4),
])
def test_grad2_kernel_vs_c_oracle(dev, B, T, V, L, seed, peaky, blocks):
    """k_grad2 forced on (it is the default only from 64 utterances on): every register-chunk variant (CH 1..16),
    several frame blocks per CTA, overlapped and serial launches -- same tolerance against the fp64 C oracle, the same
    loss bits as the k_grad path, the same gradient bits run after run and under both schedules."""
    from gluon_e2e_asr_b200 import ctc_loss_and_grad, ops
    d = make_batch(B, T, V, L, seed=seed, peaky=peaky)
    head = np.linspace(0.5, 2.0, B)
    lo, go, ok = _c_oracle(d, head=head)
    t = _to(dev, d)
    h = torch.tensor(head, device=dev, dtype=torch.float32)
    args = (t["pred"], t["label"], t["pred_lengths"], t["label_lengths"])
    with _env(grad2=0):
        ops._ws_cache.clear()
        l_old, _ = ctc_loss_and_grad(*args, head_grad=h)
        l_old = l_old.clone()
    with _env(grad2=1, grad2_blocks=blocks):
        ops._ws_cache.clear()
        loss, grad = ctc_loss_and_grad(*args, head_grad=h)
        l1, g1 = loss.clone(), grad.clone()
        loss2, grad2 = ctc_loss_and_grad(*args, head_grad=h, out_grad=torch.full_like(grad, float("nan")))
        assert torch.equal(l1, loss2) and torch.equal(g1, grad2)
        with _env(overlap=0):
            loss3, grad3 = ctc_loss_and_grad(*args, head_grad=h, out_grad=torch.full_like(grad, float("nan")))
        assert torch.equal(l1, loss3)
        torch.testing.assert_close(grad3, g1, rtol=1e-6, atol=1e-7)
    ops._ws_cache.clear()
    assert torch.equal(l1, l_old)
    _check(l1.cpu().numpy(), g1.cpu().numpy(), lo, go, "k_grad2 B=%d" % B)


def test_grad2_forward_backward_split_and_edge_cases(dev):
    """k_grad2 behind ctcb_forward(keep) / ctcb_backward (the autograd split) and on infeasible / empty utterances."""
    from gluon_e2e_asr_b200 import CtcLoss, ops
    d = make_batch(64, 120, 46, 30, seed=11)
    d["label"][1, :3] = 4; d["label_lengths"][1] = 3; d["pred_lengths"][1] = 4      # infeasible
    d["label_lengths"][2] = 0                                                         # empty label sequence
    d["pred_lengths"][3] = 0                                                          # no frames
    lo, go, ok = _c_oracle(d, head=np.full((64,), 1.0 / 64))
    t = _to(dev, d)
    with _env(grad2=1):
        ops._ws_cache.clear()
        pred = t["pred"].clone().requires_grad_(True)
        loss = CtcLoss(layout="NTC", label_layout="NT")(pred, t["label"], t["pred_lengths"], t["label_lengths"])
        loss.mean().backward()
    ops._ws_cache.clear()
    l, g = loss.detach().cpu().numpy(), pred.grad.cpu().numpy()
    assert l[1] == 0 and l[3] == 0 and not g[1].any() and not g[3].any()
    feas = [b for b in range(64) if b not in (1, 3)]
    _check(l[feas], g[feas], lo[feas], go[feas], "k_grad2 split")


def test_random_wide_vocabulary_problems_vs_c_oracle(dev):
    """Randomised wide-vocabulary problems (rows staged by bulk copies: k_emit, k_walk, the staged k_grad in every
    chunk variant, L from 0 to 200): ragged, empty and infeasible utterances, head gradients -- the fused call and
    the forward / backward split against the fp64 C oracle, status bits against its feasibility."""
    from gluon_e2e_asr_b200 import CtcLoss, ctc_loss_and_grad
    rng = np.random.default_rng(20261019)
    for case in range(36):
        B = int(rng.integers(1, 9)); T = int(rng.integers(1, 70)); V = int(rng.choice([516, 640, 1000, 2000, 3000]))
        L = int(rng.choice([0, 1, 5, 31, 32, 33, 64, 100, 129, 200]))
        lab = rng.integers(1, V, (B, max(L, 1))).astype(np.float32)
        if L > 3:
            lab[0, 1] = lab[0, 0]; lab[0, 3] = lab[0, 2]                  # repeated labels
        Lb = rng.integers(0, L + 1, B).astype(np.float32)
        Tb = rng.integers(0, T + 1, B).astype(np.float32)                # empty and infeasible utterances included
        Tb[int(rng.integers(0, B))] = T
        x = (rng.standard_normal((B, T, V)) * float(rng.choice([0.5, 2.0, 5.0]))).astype(np.float32)
        head = rng.uniform(0.25, 2.0, B)
        d = dict(pred=x, label=lab, pred_lengths=Tb, label_lengths=Lb)
        lo, go, ok = _c_oracle(d, head=head)
        t = _to(dev, d)
        status = torch.zeros((B,), dtype=torch.int32, device=dev)
        loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"],
                                       head_grad=torch.tensor(head, device=dev, dtype=torch.float32), status=status)
        name = "case %d B%d T%d V%d L%d" % (case, B, T, V, L)
        _check(loss.cpu().numpy(), grad.cpu().numpy(), lo, go, name)
        np.testing.assert_array_equal((status.cpu().numpy() & 1) == 0, ok, err_msg=name)
        if case % 3 == 0:                                                # the autograd split: k_grad on its own
            pred = t["pred"].clone().requires_grad_(True)
            l2 = CtcLoss(layout="NTC", label_layout="NT")(pred, t["label"], t["pred_lengths"], t["label_lengths"])
            (l2 * torch.tensor(head, device=dev, dtype=torch.float32)).sum().backward()
            _check(l2.detach().cpu().numpy(), pred.grad.cpu().numpy(), lo, go, name + " (split)")
