"""The operator's parameter layer on every kernel path: labels and lengths outside the documented ranges.

Five copies of the parameter layer live on the device (k_emit's metadata CTA, the fused k_walk prologue, k_meet, the
projection epilogue with its metadata kernel, k_greedy_decode).  Each must truncate and clamp labels and lengths the
same way and report the same status word.  Every path below runs one hostile batch (tests/synth.py hostile_batch) and
is checked three ways:

  (a) loss and gradient against the fp64 C oracle (rtol 1e-4 / atol 1e-5); infeasible rows exactly 0;
  (b) the whole int32 status word equals oracle.ctc_oracle.param_layer's word;
  (c) the same loss and gradient BITS as the batch clamped by hand -- only status bits 2 and 4 may differ.
"""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import ctc_oracle as O
from tests.synth import hostile_batch

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-4, 1e-5
_LIB_DT = {"i32": 0, "i64": 1, "f32": 2, "f64": 3}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _kind(a):
    return {np.float32: "f32", np.float64: "f64", np.int32: "i32", np.int64: "i64"}[np.asarray(a).dtype.type]


def _expect(d, blank_last, head=None):
    """fp64 C oracle on the clamped inputs, and param_layer's status word."""
    from oracle import ctc_ref
    B, T, V = d["pred"].shape
    bl = "last" if blank_last else "first"
    Tb, Lb, lab, st = O.param_layer(d["label"], d["pred_lengths"], d["label_lengths"], T, V, bl)
    lo, go, ok = ctc_ref.ctc_ref(d["pred"], lab, Tb, Lb, blank=V - 1 if blank_last else 0, head_grad=head,
                                 layout="NTC", dtype=np.float64)
    for b in range(B):
        go[b, Tb[b]:] = 0.0
    np.testing.assert_array_equal(ok, (st & 1) == 0)
    return lo, go, st, (Tb, Lb, lab)


def _clamped(d, clamp):
    """The same batch with its labels and lengths clamped by hand (the values the kernels must derive)."""
    Tb, Lb, lab = clamp
    return dict(pred=d["pred"], label=lab.astype(np.float32), pred_lengths=Tb.astype(np.float32),
                label_lengths=Lb.astype(np.float32))


def _dev(dev, d, tn=False):
    t = {"pred": torch.tensor(d["pred"], device=dev)}
    lab = torch.tensor(d["label"], device=dev)
    t["label"] = lab.t().contiguous() if tn else lab
    for k in ("pred_lengths", "label_lengths"):
        t[k] = None if d[k] is None else torch.tensor(d[k], device=dev)
    return t


def _fused(dev, d, blank_last, head=None, status=True, tn=False, handoff=None):
    from gluon_e2e_asr_b200 import ctc_loss_and_grad
    t = _dev(dev, d, tn)
    B = d["pred"].shape[0]
    st = torch.full((B,), -1, dtype=torch.int32, device=dev) if status else None
    h = None if head is None else torch.tensor(head, device=dev, dtype=torch.float32)
    loss, grad = ctc_loss_and_grad(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"], head_grad=h,
                                   blank_label="last" if blank_last else "first", label_layout="TN" if tn else "NT",
                                   status=st, handoff=handoff)
    torch.cuda.synchronize()
    return loss.clone(), grad.clone(), (st.cpu().numpy() if status else None)


def _check_all(name, run, d, blank_last, head=None, launches=None, grad_kernel="any", grads=True):
    """(a), (b) and (c) for one path: ``run(d) -> (loss, grad or None, status or None)`` on device tensors."""
    from gluon_e2e_asr_b200 import _lib
    lo, go, st, clamp = _expect(d, blank_last, head)
    loss, grad, status = run(d)
    if launches is not None:
        assert _lib.last_launch_count() == launches, name
    if grad_kernel != "any":
        assert _lib.last_grad_kernel() == grad_kernel, name
    l = loss.cpu().numpy()
    np.testing.assert_allclose(l, lo, rtol=RTOL, atol=ATOL, err_msg=name + " loss")
    infeasible = (st & 1) != 0
    assert infeasible.any() or d["label_lengths"] is None, name
    assert (l[infeasible] == 0).all(), name
    if grads:
        g = grad.cpu().numpy()
        np.testing.assert_allclose(g, go, rtol=RTOL, atol=ATOL, err_msg=name + " grad")
        assert (g[infeasible] == 0).all(), name
    if status is not None:
        np.testing.assert_array_equal(status, st, err_msg=name + " status word")
    # (c) the same batch clamped by hand: the same bits
    loss2, grad2, status2 = run(_clamped(d, clamp))
    assert torch.equal(loss, loss2), name + ": hostile and hand-clamped losses differ"
    if grads:
        assert torch.equal(grad, grad2), name + ": hostile and hand-clamped gradients differ"
    if status is not None:
        np.testing.assert_array_equal(status & ~6, status2 & ~6, err_msg=name)
    return loss, grad, status


def _batch(T, V, Lmax, blank_last, seed, inferred=False, **kw):
    return hostile_batch(T, V, Lmax, blank_last=blank_last, inferred=inferred, seed=seed, **kw)


# ---- the device entry: one path per shape / option ---------------------------------------------------------------------
PATHS = [
    # name, (T, V, Lmax, rows), options, launches, gradient kernel
    ("fused small V", (40, 46, 12, 1), {}, 2, "k_grad"),
    ("fused=0 dense table", (40, 46, 12, 1), {"fused": 0}, 3, "k_grad"),
    ("k_emit registers, gathered columns", (40, 300, 12, 1), {}, 3, "k_grad"),
    ("dense because V <= Lmax + 1", (250, 90, 120, 1), {}, 3, "k_grad"),
    ("staged wide rows", (40, 2000, 12, 1), {}, 3, "k_grad"),
    ("wide rows unstaged", (40, 2000, 12, 1), {"emit_staged": 0, "grad_staged": 0}, 3, "k_grad"),
    ("grad2 forced", (40, 46, 12, 1), {"grad2": 1}, 2, "k_grad2"),
    ("grad2 automatic at B >= 64", (40, 46, 12, 4), {}, 2, "k_grad2"),
    ("meet", (40, 46, 12, 1), {"meet": 1}, 1, "k_meet"),
    ("meet P=2", (40, 46, 40, 1), {"meet": 1}, 1, "k_meet"),
]


@pytest.mark.parametrize("blank_last", [False, True])
@pytest.mark.parametrize("name,shape,opts,launches,gk", PATHS, ids=[p[0] for p in PATHS])
def test_paths_clamp_and_report_like_the_oracle(dev, name, shape, opts, launches, gk, blank_last):
    from gluon_e2e_asr_b200 import _lib, ops
    T, V, Lmax, rows = shape
    if T < 2 * Lmax + 4:
        T = 2 * Lmax + 4
    with _lib.options(**opts):
        ops._ws_cache.clear()
        try:
            for inferred in (False, True):
                # (an inferred batch has 8 rows per group, a batch with lengths 18: the same B regime for both)
                d = _batch(T, V, Lmax, blank_last, seed=V + Lmax + rows, inferred=inferred,
                           rows=rows * 18 // 8 if inferred else rows)
                B = d["pred"].shape[0]
                head = np.linspace(0.5, 1.5, B)
                _check_all("%s inferred=%s" % (name, inferred), lambda x: _fused(dev, x, blank_last, head), d,
                           blank_last, head, launches, gk)
        finally:
            ops._ws_cache.clear()


@pytest.mark.parametrize("meet_fwd", [0, 1])
@pytest.mark.parametrize("blank_last", [False, True])
def test_forward_only(dev, meet_fwd, blank_last):
    """Loss evaluation without a gradient: the recursion kernel alone (V = 46) or behind k_emit (V = 300), one walker per
    utterance (meet_fwd=0) or an alpha and a beta walker that meet in the middle (meet_fwd=1)."""
    from gluon_e2e_asr_b200 import _lib, ops

    def run(x):
        t = _dev(dev, x)
        call = ops._Call(t["pred"], t["label"], t["pred_lengths"], t["label_lengths"], blank_last, True, False)
        loss = torch.full((call.B,), float("nan"), device=dev)
        st = torch.full((call.B,), -1, dtype=torch.int32, device=dev)
        ws = ops._alloc_ws(call, False)
        call.run(_lib.PHASE_FORWARD, ws, loss, status=st)
        torch.cuda.synchronize()
        return loss, None, st.cpu().numpy()

    with _lib.options(meet_fwd=meet_fwd):
        for V in (46, 300):
            for inferred in (False, True):
                d = _batch(40, V, 12, blank_last, seed=5 + V, inferred=inferred)
                _check_all("forward only V=%d meet_fwd=%d" % (V, meet_fwd), run, d, blank_last, launches=1 if V <= 64 else 2,
                           grad_kernel=None, grads=False)


def test_autograd_split_and_handoffs(dev):
    """The autograd split (history kept in Forward, gradient in Backward) and both hand-offs (DLPack is used only without
    a status vector) against the oracle, with the same bits as the fused call that reports status."""
    from gluon_e2e_asr_b200 import CtcLoss, ops
    for blank_last in (False, True):
        bl = "last" if blank_last else "first"
        for V in (46, 300):
            d = _batch(40, V, 12, blank_last, seed=11 + V)
            B = d["pred"].shape[0]
            head = np.linspace(0.5, 1.5, B)
            loss, grad, _ = _check_all("status call V=%d" % V, lambda x: _fused(dev, x, blank_last, head), d, blank_last, head)
            for handoff in ("dlpack", "pointer"):
                l2, g2, _ = _fused(dev, d, blank_last, head, status=False, handoff=handoff)
                assert torch.equal(l2, loss) and torch.equal(g2, grad), handoff

            def split(x):
                t = _dev(dev, x)
                pred = t["pred"].clone().requires_grad_(True)
                l = CtcLoss(layout="NTC", label_layout="NT", blank_label=bl)(pred, t["label"], t["pred_lengths"],
                                                                            t["label_lengths"])
                (l * torch.tensor(head, device=dev, dtype=torch.float32)).sum().backward()
                return l.detach(), pred.grad, None

            saved = ops._FUSE_IN_FORWARD_MAX_ELEMS
            try:
                ops._FUSE_IN_FORWARD_MAX_ELEMS = 0
                _check_all("autograd split V=%d" % V, split, d, blank_last, head)
            finally:
                ops._FUSE_IN_FORWARD_MAX_ELEMS = saved


def _host_problem(x, blank_last, status, loss, grad=None):
    """ctcb_problem_t over host numpy buffers of a batch (NTC logits, NT labels)."""
    from gluon_e2e_asr_b200 import _lib
    B, T, V = x["pred"].shape
    Lmax = x["label"].shape[1]
    p = _lib.Problem()
    p.T, p.B, p.V, p.Lmax = T, B, V, Lmax
    p.blank, p.label_pad = (V - 1, -1) if blank_last else (0, 0)
    p.logits, p.logits_stride_t, p.logits_stride_b = x["pred"].ctypes.data, V, T * V
    if grad is not None:
        p.grad, p.grad_stride_t, p.grad_stride_b = grad.ctypes.data, V, T * V
    p.labels, p.label_dtype, p.label_stride_b, p.label_stride_l = x["label"].ctypes.data, _LIB_DT[_kind(x["label"])], Lmax, 1
    p.data_lengths, p.data_lengths_dtype = x["pred_lengths"].ctypes.data, _LIB_DT[_kind(x["pred_lengths"])]
    if x["label_lengths"] is not None:
        p.label_lengths, p.label_lengths_dtype = x["label_lengths"].ctypes.data, _LIB_DT[_kind(x["label_lengths"])]
    p.loss, p.status = loss.ctypes.data, status.ctypes.data
    return p


def test_host_entry_and_pipeline(dev):
    """ctcb_loss_grad_host (host buffers in and out) and HostPipeline with a dense and a packed PinnedBatch."""
    from gluon_e2e_asr_b200 import HostPipeline, PinnedBatch, _lib
    for blank_last in (False, True):
        for inferred in (False, True):
            d = _batch(40, 46, 12, blank_last, seed=21, inferred=inferred, label_dtype="f32", length_dtype="f64")
            B = d["pred"].shape[0]

            def host(x):
                x = {k: (None if v is None else np.ascontiguousarray(v)) for k, v in x.items()}
                loss = np.full((B,), np.nan, np.float32); st = np.full((B,), -1, np.int32)
                g = np.full_like(x["pred"], np.nan)
                p = _host_problem(x, blank_last, st, loss, g)
                _lib.check(_lib.load().ctcb_loss_grad_host(ctypes.byref(p), 0))
                return torch.tensor(loss), torch.tensor(g), st

            _check_all("host entry inferred=%s" % inferred, host, d, blank_last)
            if inferred:
                continue                                   # PinnedBatch carries both length vectors
            for packed in (False, True):
                pipe = HostPipeline(0, depth=2)
                try:
                    def piped(x):
                        pb = PinnedBatch.from_arrays(x["pred"], x["label"], x["pred_lengths"], x["label_lengths"],
                                                     packed=packed)
                        lo = torch.full((B,), float("nan")).pin_memory()
                        st = np.full((B,), -1, np.int32)
                        q = pipe.problem(pb, lo, "last" if blank_last else "first")
                        q.status = st.ctypes.data
                        g = pipe.wait(pipe.submit_problem(q))
                        return lo.clone(), g.clone(), st

                    _check_all("pipeline packed=%s" % packed, piped, d, blank_last)
                finally:
                    pipe.close()


@pytest.mark.parametrize("V", [300, 600])
@pytest.mark.parametrize("blank_last", [False, True])
def test_fused_projection(dev, V, blank_last):
    """ctcb_proj_loss_grad with a status vector: the projection epilogue clamps labels and frame counts itself and the
    metadata kernel beside it reports the status word.  Operands exact in tf32, so the fp64 product is the logits."""
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _Call, _alloc_ws, _stream_ptr
    from gluon_e2e_asr_b200.proj import _proj_struct
    T, K, Lmax = 150, 64, 12
    tf32 = lambda a: (np.ascontiguousarray(a, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
    for inferred in (False, True):
        d = _batch(T, V, Lmax, blank_last, seed=V + 7, inferred=inferred)
        B = d["pred"].shape[0]
        rng = np.random.Generator(np.random.PCG64(V))
        h = tf32(rng.standard_normal((B, T, K)))
        w = tf32(rng.standard_normal((V, K)) / np.sqrt(K))
        bv = (rng.standard_normal((V,)) * 0.5).astype(np.float32)
        d["pred"] = (h.astype(np.float64) @ w.astype(np.float64).T + bv).astype(np.float32)
        head = np.linspace(0.5, 1.5, B)
        th, tw, tb = (torch.tensor(a, device=dev) for a in (h, w, bv))
        logits64 = h.astype(np.float64) @ w.astype(np.float64).T + bv

        def run(x):
            t = _dev(dev, x)
            logits = torch.full((B, T, V), float("nan"), device=dev)
            grad = torch.full_like(logits, float("nan"))
            loss = torch.full((B,), float("nan"), device=dev)
            st = torch.full((B,), -1, dtype=torch.int32, device=dev)
            call = _Call(logits, t["label"], t["pred_lengths"], t["label_lengths"], blank_last, True, False)
            ws = _alloc_ws(call, True)
            p = call.problem(loss, grad, torch.tensor(head, device=dev, dtype=torch.float32), status=st)
            _lib.check(_lib.load().ctcb_proj_loss_grad(ctypes.byref(_proj_struct(th, tw, tb)), ctypes.byref(p),
                                                       ws.data_ptr(), ws.numel(), _stream_ptr(dev)))
            torch.cuda.synchronize()
            return loss, grad, st.cpu().numpy()

        # the oracle of the fp64 product (the kernel's tf32 products of tf32-exact operands, fp32 accumulation)
        from oracle import ctc_ref
        bl = "last" if blank_last else "first"
        Tb, Lb, lab, st = O.param_layer(d["label"], d["pred_lengths"], d["label_lengths"], T, V, bl)
        lo, go, ok = ctc_ref.ctc_ref(logits64, lab, Tb, Lb, blank=V - 1 if blank_last else 0, head_grad=head,
                                     layout="NTC", dtype=np.float64)
        for b in range(B):
            go[b, Tb[b]:] = 0.0
        loss, grad, status = run(d)
        assert _lib.last_launch_count() == 4
        np.testing.assert_array_equal(status, st, err_msg="projection status word")
        np.testing.assert_allclose(loss.cpu().numpy(), lo, rtol=RTOL, atol=ATOL, err_msg="projection loss")
        np.testing.assert_allclose(grad.cpu().numpy(), go, rtol=RTOL, atol=ATOL, err_msg="projection d logits")
        loss2, grad2, status2 = run(_clamped(d, (Tb, Lb, lab)))
        assert torch.equal(loss, loss2) and torch.equal(grad, grad2)
        np.testing.assert_array_equal(status & ~6, status2 & ~6)


def test_label_and_length_dtypes_give_the_same_bits(dev):
    """Labels in f32/f64/i32/i64 x lengths in f32/f64/i32/i64, NT and TN label layouts: the same loss, gradient and status
    bits (fractional values only in the float dtypes; each integer dtype carries its own huge values)."""
    for blank_last in (False, True):
        for inferred in (False, True):
            ref = None
            for ld in ("f32", "f64", "i32", "i64"):
                for nd in ("f32", "f64", "i32", "i64"):
                    d = _batch(40, 46, 12, blank_last, seed=33, inferred=inferred, label_dtype=ld, length_dtype=nd)
                    for tn in (False, True):
                        got = _fused(dev, d, blank_last, tn=tn)
                        if ref is None:
                            lo, go, st, _ = _expect(d, blank_last)
                            np.testing.assert_allclose(got[0].cpu().numpy(), lo, rtol=RTOL, atol=ATOL)
                            np.testing.assert_allclose(got[1].cpu().numpy(), go, rtol=RTOL, atol=ATOL)
                            np.testing.assert_array_equal(got[2], st)
                            ref = got
                        where = "labels %s lengths %s TN=%s blank_last=%s inferred=%s" % (ld, nd, tn, blank_last, inferred)
                        assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1]), where
                        np.testing.assert_array_equal(got[2], ref[2], err_msg=where)


@pytest.mark.parametrize("V", [46, 2000])
def test_greedy_decode_clamps_lengths(dev, V):
    """k_greedy_decode: frame counts negative, beyond T and fractional, in all four dtypes, against the oracle (which
    truncates and clamps them to [0, T]); with and without the <unk> rule."""
    from gluon_e2e_asr_b200 import greedy_decode
    B, T = 8, 60
    rng = np.random.default_rng(V)
    x = rng.standard_normal((B, T, V)).astype(np.float32)
    x[:, ::3, 0] += 4.0                                        # blanks between symbols
    master = np.array([-3, T + 9, 17.9, T, 0, -0.5, np.inf, 33.2])
    from tests.synth import _cast
    xt = torch.tensor(x, device=dev)
    for kind in ("f32", "f64", "i32", "i64"):
        lens = _cast(master, kind)
        for unk in (None, 5):
            toks, n = greedy_decode(xt, torch.tensor(lens, device=dev), unk=unk)
            ref = O.greedy_decode(x, lens) if unk is None else O.greedy_decode_unk(x, lens, unk)
            toks, n = toks.cpu().numpy(), n.cpu().numpy()
            for b in range(B):
                assert list(toks[b, :n[b]]) == ref[b], (kind, unk, b)
            assert n[0] == 0 and n[4] == 0 and n[5] == 0
