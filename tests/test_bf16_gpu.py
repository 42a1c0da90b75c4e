"""bfloat16 logits on the device loss path (include/ctcb.h, the *_typed entries).

The contract: a bf16 logit is widened to fp32 exactly when it is loaded and everything after that is the fp32 path's.
So the bf16 call and the fp32 call on ``x_bf16.float()`` must pick the same kernels, give the same loss bits and status
word, and the bf16 gradient must be the fp32 gradient rounded once to bf16 -- bit for bit.  On top of that the results
are checked against the fp64 oracle on the upcast values (loss at the fp32 bar, gradient with one bf16 rounding more).
"""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import ctc_oracle as O
from tests.synth import CONFIGS, hostile_batch, make_batch
from tests.test_param_layer_gpu import PATHS, _expect

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-4, 1e-5
GRAD_RTOL = 2.0 ** -8 + RTOL          # one bf16 rounding (<= 2^-8 relative) on top of the fp32 bar

# every path of the fp32 tests except the opt-in one-kernel path (fp32 only; see test_meet_option_takes_two_kernels)
BF_PATHS = [p for p in PATHS if p[4] != "k_meet"]


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


def _labels(dev, d):
    t = {"label": torch.tensor(d["label"], device=dev)}
    for k in ("pred_lengths", "label_lengths"):
        t[k] = None if d[k] is None else torch.tensor(d[k], device=dev)
    return t


def _upcast(d, xb):
    """The batch with its logits replaced by the bf16 values, widened (what the oracle and the fp32 arm see)."""
    e = dict(d)
    e["pred"] = xb.float().cpu().numpy()
    return e


def _step(x, t, blank_last, layout, head, handoff, status):
    """One fused call; returns (loss, grad, status or None, (launches, gradient kernel, walker configuration))."""
    from gluon_e2e_asr_b200 import _lib, ctc_loss_and_grad
    B = t["label"].shape[0]
    st = torch.full((B,), -1, dtype=torch.int32, device=x.device) if status else None
    h = None if head is None else torch.tensor(head, device=x.device, dtype=torch.float32)
    loss, grad = ctc_loss_and_grad(x, t["label"], t["pred_lengths"], t["label_lengths"], head_grad=h,
                                   blank_label="last" if blank_last else "first", layout=layout, status=st, handoff=handoff)
    torch.cuda.synchronize()
    kern = (_lib.last_launch_count(), _lib.last_grad_kernel(), _lib.last_walk_config())
    return loss.clone(), grad.clone(), (st.cpu().numpy() if status else None), kern


def _ntc(g, layout):
    return g if layout == "NTC" else g.transpose(0, 1)


@pytest.mark.parametrize("blank_last", [False, True])
@pytest.mark.parametrize("name,shape,opts,launches,gk", BF_PATHS, ids=[p[0] for p in BF_PATHS])
def test_paths_bit_for_bit(dev, name, shape, opts, launches, gk, blank_last):
    """Each kernel path: bf16 against fp32 on the upcast logits (kernels, loss bits, status, gradient rounded once), NTC and
    TNC, with and without head gradients, both hand-offs and with status; then against the fp64 oracle."""
    from gluon_e2e_asr_b200 import _lib, ops
    T, V, Lmax, rows = shape
    T = max(T, 2 * Lmax + 4)
    with _lib.options(**opts):
        ops._ws_cache.clear()
        try:
            d = hostile_batch(T, V, Lmax, blank_last=blank_last, seed=V + Lmax + rows, rows=rows)
            B = d["pred"].shape[0]
            t = _labels(dev, d)
            xb_ntc = torch.tensor(d["pred"], device=dev).to(torch.bfloat16)
            du = _upcast(d, xb_ntc)
            for layout in ("NTC", "TNC"):
                xb = xb_ntc if layout == "NTC" else xb_ntc.transpose(0, 1).contiguous()
                xf = xb.float()
                for head in (None, np.linspace(0.5, 1.5, B)):
                    lo, go, st_o, _ = _expect(du, blank_last, head)
                    for handoff, status in (("dlpack", False), ("pointer", False), ("pointer", True)):
                        what = "%s %s head=%s %s status=%s" % (name, layout, head is not None, handoff, status)
                        lb, gb, sb, kb = _step(xb, t, blank_last, layout, head, handoff, status)
                        lf, gf, sf, kf = _step(xf, t, blank_last, layout, head, handoff, status)
                        assert kb == kf, what
                        assert kb[0] == launches and kb[1] == gk, (what, kb)
                        assert lb.dtype == torch.float32 and gb.dtype == torch.bfloat16, what
                        assert torch.equal(_bits(lb), _bits(lf)), what + ": loss bits"
                        assert torch.equal(_bits(gb), _bits(gf.to(torch.bfloat16))), what + ": gradient not fp32 rounded once"
                        if status:
                            np.testing.assert_array_equal(sb, sf, err_msg=what)
                            np.testing.assert_array_equal(sb, st_o, err_msg=what)
                        # against the oracle on the upcast values
                        l = lb.cpu().numpy()
                        g = _ntc(gb, layout).float().cpu().numpy()
                        infeasible = (st_o & 1) != 0
                        np.testing.assert_allclose(l, lo, rtol=RTOL, atol=ATOL, err_msg=what + " loss")
                        np.testing.assert_allclose(g, go, rtol=GRAD_RTOL, atol=ATOL, err_msg=what + " grad")
                        assert (l[infeasible] == 0).all() and (g[infeasible] == 0).all(), what
        finally:
            ops._ws_cache.clear()


@pytest.mark.parametrize("meet_fwd", [0, 1])
@pytest.mark.parametrize("blank_last", [False, True])
def test_forward_only_bits(dev, meet_fwd, blank_last):
    """Loss evaluation (both walker schedules, with and without k_emit): loss and status bits of the fp32 call."""
    from gluon_e2e_asr_b200 import _lib, ops

    def run(x, t):
        call = ops._Call(x, t["label"], t["pred_lengths"], t["label_lengths"], blank_last, True, False)
        loss = torch.full((call.B,), float("nan"), device=dev)
        st = torch.full((call.B,), -1, dtype=torch.int32, device=dev)
        call.run(_lib.PHASE_FORWARD, ops._alloc_ws(call, False), loss, status=st)
        torch.cuda.synchronize()
        return loss, st.cpu().numpy(), _lib.last_launch_count()

    with _lib.options(meet_fwd=meet_fwd):
        for V in (46, 300, 2000):
            d = hostile_batch(40, V, 12, blank_last=blank_last, seed=5 + V)
            t = _labels(dev, d)
            xb = torch.tensor(d["pred"], device=dev).to(torch.bfloat16)
            lb, sb, nb = run(xb, t)
            lf, sf, nf = run(xb.float(), t)
            assert nb == nf
            assert torch.equal(_bits(lb), _bits(lf)), V
            np.testing.assert_array_equal(sb, sf)
            lo, _, st_o, _ = _expect(_upcast(d, xb), blank_last)
            np.testing.assert_allclose(lb.cpu().numpy(), lo, rtol=RTOL, atol=ATOL)
            np.testing.assert_array_equal(sb, st_o)


@pytest.mark.parametrize("V", [46, 2000])
def test_autograd_returns_bf16_gradient(dev, V):
    """CtcLoss on a bf16 tensor: fp32 loss, bf16 gradient equal to the fp32 keep-history path's gradient rounded once."""
    from gluon_e2e_asr_b200 import CtcLoss, ops
    d = make_batch(8, 120, V, 20, seed=3)
    t = _labels(dev, d)
    xb = torch.tensor(d["pred"], device=dev).to(torch.bfloat16)

    def step(x):
        pred = x.clone().requires_grad_(True)
        loss = CtcLoss(layout="NTC", label_layout="NT")(pred, t["label"], t["pred_lengths"], t["label_lengths"])
        loss.mean().backward()
        torch.cuda.synchronize()
        return loss.detach(), pred.grad

    lb, gb = step(xb)
    assert lb.dtype == torch.float32 and gb.dtype == torch.bfloat16
    saved = ops._FUSE_IN_FORWARD_MAX_ELEMS
    try:
        ops._FUSE_IN_FORWARD_MAX_ELEMS = 0
        lf, gf = step(xb.float())
    finally:
        ops._FUSE_IN_FORWARD_MAX_ELEMS = saved
    assert torch.equal(_bits(lb), _bits(lf))
    assert torch.equal(_bits(gb), _bits(gf.to(torch.bfloat16)))
    lo, go, _ = O.CtcLossOracle("NTC", "NT")(_upcast(d, xb)["pred"], d["label"], d["pred_lengths"], d["label_lengths"],
                                             head_grad=np.full((8,), 1.0 / 8))
    np.testing.assert_allclose(lb.cpu().numpy(), lo, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(gb.float().cpu().numpy(), go, rtol=GRAD_RTOL, atol=ATOL)


def _oracle_check(l, g, du, blank_last=False, head=None, what=""):
    lo, go, st_o, _ = _expect(du, blank_last, head)
    np.testing.assert_allclose(l, lo, rtol=RTOL, atol=ATOL, err_msg=what + " loss")
    np.testing.assert_allclose(g, go, rtol=GRAD_RTOL, atol=ATOL, err_msg=what + " grad")
    infeasible = (st_o & 1) != 0
    assert (l[infeasible] == 0).all() and (g[infeasible] == 0).all(), what


@pytest.mark.parametrize("V", [46, 2000])
def test_packed_rows(dev, V):
    """logits_row_offsets (packed rows, only the valid frames stored) with bf16 logits, against the oracle and against the
    fp32 call on the same packed values."""
    from gluon_e2e_asr_b200 import _lib, ops
    d = hostile_batch(40, V, 12, seed=21 + V)
    B, T, _ = d["pred"].shape
    t = _labels(dev, d)
    xb = torch.tensor(d["pred"], device=dev).to(torch.bfloat16)
    Tb = np.clip(np.trunc(d["pred_lengths"]).astype(np.int64), 0, T)
    offs = np.concatenate([[0], np.cumsum(Tb[:-1] * V)]).astype(np.int64)

    def run(x):
        packed = torch.cat([x[b, :Tb[b]].reshape(-1) for b in range(B)] + [x.new_zeros(V)])
        call = ops._Call(x, t["label"], t["pred_lengths"], t["label_lengths"], False, True, False)
        loss = torch.empty((B,), device=dev)
        grad = torch.full_like(x, float("nan"))
        off_t = torch.tensor(offs, device=dev)
        p = call.problem(loss, grad)
        p.logits, p.logits_row_offsets = packed.data_ptr(), off_t.data_ptr()
        ws = ops._alloc_ws(call, True)
        with torch.cuda.device(dev):
            rc = _lib.load().ctcb_loss_grad_typed(ctypes.byref(p), call.ldt, ws.data_ptr(), ws.numel(),
                                                  ops._stream_ptr(dev))
        _lib.check(rc)
        torch.cuda.synchronize()
        return loss, grad

    lb, gb = run(xb)
    lf, gf = run(xb.float())
    assert torch.equal(_bits(lb), _bits(lf))
    assert torch.equal(_bits(gb), _bits(gf.to(torch.bfloat16)))
    _oracle_check(lb.cpu().numpy(), gb.float().cpu().numpy(), _upcast(d, xb), what="packed V=%d" % V)


@pytest.mark.parametrize("V", [47, 301])
def test_odd_vocabulary_and_strided_rows(dev, V):
    """An odd V (one-element loads) and a strided view of a wider buffer, bf16 against fp32 and the oracle."""
    d = hostile_batch(40, V, 12, seed=31 + V)
    B, T, _ = d["pred"].shape
    t = _labels(dev, d)
    wide = torch.zeros((B, T, V + 3), device=dev, dtype=torch.bfloat16)
    wide[:, :, 1:V + 1] = torch.tensor(d["pred"], device=dev).to(torch.bfloat16)
    for xb in (wide[:, :, 1:V + 1].contiguous(), wide[:, :, 1:V + 1]):
        lb, gb, _, kb = _step(xb, t, False, "NTC", None, "pointer", False)
        lf, gf, _, kf = _step(xb.float(), t, False, "NTC", None, "pointer", False)
        assert kb == kf
        assert torch.equal(_bits(lb), _bits(lf))
        assert torch.equal(_bits(gb), _bits(gf.to(torch.bfloat16)))
        _oracle_check(lb.cpu().numpy(), gb.float().cpu().numpy(), _upcast(d, xb), what="V=%d" % V)


def test_meet_option_takes_two_kernels(dev):
    """The one-kernel path is fp32-only: with meet=1 a bf16 call runs k_walk + k_grad and still matches the oracle."""
    from gluon_e2e_asr_b200 import _lib, ops
    d = hostile_batch(40, 46, 12, seed=7)
    t = _labels(dev, d)
    xb = torch.tensor(d["pred"], device=dev).to(torch.bfloat16)
    with _lib.options(meet=1):
        ops._ws_cache.clear()
        try:
            lf, gf, _, kf = _step(xb.float(), t, False, "NTC", None, "pointer", True)
            assert kf[1] == "k_meet"
            lb, gb, sb, kb = _step(xb, t, False, "NTC", None, "pointer", True)
        finally:
            ops._ws_cache.clear()
    assert kb[1] != "k_meet" and kb[0] == 2
    _oracle_check(lb.cpu().numpy(), gb.float().cpu().numpy(), _upcast(d, xb), what="meet=1")


def test_refusals(dev):
    from gluon_e2e_asr_b200 import _lib, ctc_loss_and_grad, greedy_decode, ops
    d = make_batch(2, 30, 46, 5, seed=1)
    t = _labels(dev, d)
    x16 = torch.tensor(d["pred"], device=dev).to(torch.float16)
    with pytest.raises(TypeError, match="float16"):
        ctc_loss_and_grad(x16, t["label"], t["pred_lengths"], t["label_lengths"])
    with pytest.raises(TypeError, match="float16"):
        greedy_decode(x16)
    xb = x16.to(torch.bfloat16)
    with pytest.raises(TypeError, match="out_grad"):
        ctc_loss_and_grad(xb, t["label"], t["pred_lengths"], t["label_lengths"], out_grad=torch.empty_like(xb, dtype=torch.float32))
    # the DLPack entry checks the gradient tensor's dtype itself
    call = ops._Call(xb, t["label"], t["pred_lengths"], t["label_lengths"], False, True, False)
    loss = torch.empty((2,), device=dev)
    for wrong in (torch.float32, torch.float16):
        with pytest.raises(_lib.CtcbError) as e:
            call.run(_lib.PHASE_FUSED, ops._alloc_ws(call, True), loss, grad=torch.empty_like(xb, dtype=wrong), handoff="dlpack")
        assert e.value.code == _lib.CTCB_INVALID_VALUE and "dtype" in str(e.value)
    # fp32 logits with a bf16 gradient tensor: refused the same way
    call32 = ops._Call(xb.float(), t["label"], t["pred_lengths"], t["label_lengths"], False, True, False)
    with pytest.raises(_lib.CtcbError):
        call32.run(_lib.PHASE_FUSED, ops._alloc_ws(call32, True), loss, grad=torch.empty_like(xb), handoff="dlpack")


@pytest.mark.parametrize("V", [46, 2000])
def test_greedy_decode_ties(dev, V):
    """bf16 decode equals the oracle decode of the upcast values, with and without <unk>, on logits full of exact ties
    (a handful of distinct values per frame: the lowest index must win)."""
    from gluon_e2e_asr_b200 import greedy_decode
    B, T = 8, 80
    rng = np.random.default_rng(V + 1)
    x = (rng.integers(-2, 3, (B, T, V)) * 0.5).astype(np.float32)          # exact in bf16, ties everywhere
    x[:, ::4, 0] += 1.0
    x[:, 1::5, 7] = x[:, 1::5].max(axis=-1)                                 # a tie of <unk> with a lower and a higher index
    x[:, 2::7, 5] = x[:, 2::7].max(axis=-1) + 0.5
    lens = np.array([T, T - 3, 17, 0, T, 40, 1, T], np.float32)
    xb = torch.tensor(x, device=dev).to(torch.bfloat16)
    xu = xb.float().cpu().numpy()
    assert np.array_equal(xu, x)
    for unk in (None, 5, 7):
        toks, n = greedy_decode(xb, torch.tensor(lens, device=dev), unk=unk)
        ref = O.greedy_decode(xu, lens) if unk is None else O.greedy_decode_unk(xu, lens, unk)
        toks, n = toks.cpu().numpy(), n.cpu().numpy()
        for b in range(B):
            assert list(toks[b, :n[b]]) == ref[b], (unk, b)
        # the same tokens as the fp32 decode
        t32, n32 = greedy_decode(xb.float(), torch.tensor(lens, device=dev), unk=unk)
        assert torch.equal(t32, torch.tensor(toks, device=dev)) and torch.equal(n32.cpu(), torch.tensor(n))


def test_config_shapes_pick_the_same_kernels(dev):
    """cfg1-cfg5 (the benchmark's shapes, fresh contiguous tensors): the bf16 call selects the kernels of the fp32 call --
    cfg3 included, whose bf16 rows (V * 2 = 4000 bytes) take the staged (bulk-copy) gradient kernel like fp32 ones."""
    from gluon_e2e_asr_b200 import _lib
    for name, (B, T, V, L) in CONFIGS.items():
        d = make_batch(B, T, V, L, seed=0)
        t = _labels(dev, d)
        xb = torch.tensor(d["pred"], device=dev).to(torch.bfloat16)
        lb, gb, _, kb = _step(xb, t, False, "NTC", None, "pointer", False)
        lf, gf, _, kf = _step(xb.float(), t, False, "NTC", None, "pointer", False)
        assert kb == kf, name
        assert torch.equal(_bits(lb), _bits(lf)), name
        assert torch.equal(_bits(gb), _bits(gf.to(torch.bfloat16))), name
        del lb, gb, lf, gf
