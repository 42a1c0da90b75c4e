"""Every kernel path on memory it did not get clean.

The workspace is caller-owned scratch: torch's caching allocator hands back whatever the last tensor in the block held,
and a caller may size one buffer for its largest bucket and share it between calls on one stream.  include/ctcb.h
promises that its contents on entry do not matter.  Each row of ROWS (a kernel path, pinned to its launches, gradient
kernel and walker configuration) runs on a workspace in six states:

  zero    all bytes 0 -- the reference run, checked against the fp64 C oracle;
  ff      all bytes 0xFF: int -1, a NaN double, sign bits set;
  7f      all bytes 0x7F: huge positive counters and values;
  random  seeded random bytes;
  other   what a different problem left (a larger Lmax, the other vocabulary class, automatic options), enqueued just
          before, no sync;
  same    what the same shape with other logits and labels left: the same stamp, so the progress words look complete.
The last two start from a buffer of 0xA5 bytes, which the earlier call then partly overwrites.

Loss, gradient (or G), status word, tokens and lengths must have the zero run's bits; loss_sum (fp64 atomics, not
bit-reproducible) agrees to 1e-12 relative.  Then: one buffer shared by a bucketed loop of mixed problems, in both orders;
graph replays whose workspace is overwritten between replays; and padded frames / label slots / hidden rows filled with
NaN, infinities and huge values, which must give the bits of the zero-padded batch."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import ctc_oracle as O
from tests.synth import make_batch
from tests.test_param_layer_gpu import _expect
from tests.test_proj_recompute_edges_gpu import _logits64, _oracle, _weights

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-4, 1e-5
GRAD_RTOL_BF16 = 2.0 ** -8 + RTOL          # one bf16 rounding of the gradient on top of the fp32 bar
NAN = float("nan")
STATES = ("zero", "ff", "7f", "random", "other", "same")
PAD_LOGITS = (NAN, float("inf"), -float("inf"), 3e38, -3e38)
PAD_LABELS = (1e10, -7.0, NAN)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


class Row:
    """One kernel path: an entry point, a shape and the options that select it, and what each of its C calls launches:
    ``kern`` = [(launches, gradient kernel or "any", walker configuration or None), ...] in call order."""

    def __init__(self, name, entry, B, T, V, L, kern, opts=None, bf16=False, K=0, ctas=2):
        self.name, self.entry, self.B, self.T, self.V, self.L = name, entry, B, T, V, L
        self.kern, self.opts, self.bf16, self.K, self.ctas = kern, dict(opts or {}), bf16, K, ctas
        if entry.startswith("proj"):
            self.opts.setdefault("proj_ctas", ctas)

    @property
    def proj(self):
        return self.entry.startswith("proj")

    @property
    def need_grad(self):
        return self.entry in ("loss_grad", "split", "proj_loss_grad", "proj_recompute")

    def ws_bytes(self):
        from gluon_e2e_asr_b200 import _lib
        return _lib.workspace_bytes(self.T, self.B, self.V, self.L, self.need_grad)


def _T(L, lo=40):
    return max(lo, 2 * L + 40)


def _loss(name, B, V, L, kern, T=None, **kw):
    return Row(name, kw.pop("entry", "loss_grad"), B, T or _T(L), V, L, kern, **kw)


G1, G2, MEET = "k_grad", "k_grad2", "k_meet"
# Batch of the rows whose gradient CTAs run beside the fused walkers.  Stale progress words are only visible to gradient
# CTAs that reach a frame block before its walker does, which is a matter of timing.  Measured on B200 with the walkers'
# reset of their progress words removed: 1 of 30 runs on 0x7F or same-shape workspaces showed the stale history at 3
# utterances, 14 of 15 at 16 (L = 200); a whole run of this file failed the two L = 200 rows at 16 utterances.
BO = 16
ROWS = [
    # the fused path (V <= 64): k_walk fused + k_grad, every chunk count of the gradient kernel
    _loss("fused L12 CH1", BO, 46, 12, [(2, G1, (1, 1))]),
    _loss("fused L100 CH4", BO, 46, 100, [(2, G1, (2, 2))]),
    _loss("fused L200 CH8", BO, 46, 200, [(2, G1, (2, 4))]),
    _loss("fused L400 CH16", BO, 46, 400, [(2, G1, (2, 8))]),
    _loss("fused V30 L700 CH0", BO, 30, 700, [(2, G1, (2, 12))]),
    # k_grad2: the chunk variants of the blank-column guard, and its automatic choice
    _loss("grad2 L12 CH1", BO, 46, 12, [(2, G2, (1, 1))], opts={"grad2": 1}),
    _loss("grad2 L100 CH4", BO, 46, 100, [(2, G2, (2, 2))], opts={"grad2": 1}),
    _loss("grad2 L200 CH8", BO, 46, 200, [(2, G2, (2, 4))], opts={"grad2": 1}),
    _loss("grad2 L400 CH16", BO, 46, 400, [(2, G2, (2, 8))], opts={"grad2": 1}),
    _loss("grad2 automatic B64", 64, 46, 12, [(2, G2, (1, 1))]),
    # serial variants: the gradient kernel runs after the walkers
    _loss("B320 grad2 plain launch", 320, 46, 12, [(2, G2, (1, 1))]),
    _loss("B320 V300 high-occupancy k_grad", 320, 300, 12, [(3, G1, (1, 1))]),
    _loss("overlap=0", 3, 46, 12, [(2, G1, (1, 1))], opts={"overlap": 0}),
    _loss("grad2 grad2_occ=0", BO, 46, 100, [(2, G2, (2, 2))], opts={"grad2": 1, "grad2_occ": 0}),
    # wide vocabularies, register variants of k_emit / k_grad
    _loss("wide V90 VEC2", 3, 90, 12, [(3, G1, (1, 1))]),
    _loss("wide V301 VEC1", 3, 301, 12, [(3, G1, (1, 1))]),
    _loss("wide V300 VEC4", 3, 300, 12, [(3, G1, (1, 1))]),
    _loss("dense V90 L120", 3, 90, 120, [(3, G1, (2, 2))]),
    # wide vocabularies, staged and unstaged rows; k_grad CH 8 / 16 / 0 on the plain device entry
    _loss("wide V2000 L150", 2, 2000, 150, [(3, G1, (2, 3))]),
    _loss("wide V2000 L300", 2, 2000, 300, [(3, G1, (2, 5))]),
    _loss("wide V2000 L600", 2, 2000, 600, [(3, G1, (2, 12))]),
    _loss("wide V2000 L150 unstaged", 2, 2000, 150, [(3, G1, (2, 3))], opts={"emit_staged": 0, "grad_staged": 0}),
    _loss("wide V2000 L600 unstaged", 2, 2000, 600, [(3, G1, (2, 12))], opts={"emit_staged": 0, "grad_staged": 0}),
    # the one-kernel path
    _loss("meet P1", 3, 46, 12, [(1, MEET, (1, 1))], opts={"meet": 1}),
    _loss("meet P2", 3, 46, 40, [(1, MEET, (2, 1))], opts={"meet": 1}),
    _loss("meet P4", 3, 46, 100, [(1, MEET, (4, 1))], opts={"meet": 1}),
    # loss evaluation: one walker per utterance, or two that meet in the middle (meetcnt)
    _loss("forward V46 meet_fwd=0", 3, 46, 30, [(1, None, (1, 1))], entry="forward", opts={"meet_fwd": 0}),
    _loss("forward V46 meet_fwd=1", 3, 46, 30, [(1, None, (1, 1))], entry="forward", opts={"meet_fwd": 1}),
    _loss("forward V300 meet_fwd=0", 3, 300, 30, [(2, None, (1, 1))], entry="forward", opts={"meet_fwd": 0}),
    _loss("forward V300 meet_fwd=1", 3, 300, 30, [(2, None, (1, 1))], entry="forward", opts={"meet_fwd": 1}),
    # the autograd split: dirty state before the forward only (the buffer is the history in between)
    _loss("split V46", 3, 46, 50, [(1, None, (2, 1)), (1, G1, None)], entry="split"),
    _loss("split V300", 3, 300, 50, [(2, None, (2, 1)), (1, G1, None)], entry="split"),
    # bfloat16 logits
    _loss("bf16 V46 L200", BO, 46, 200, [(2, G1, (2, 4))], bf16=True),
    _loss("bf16 grad2 L200", BO, 46, 200, [(2, G2, (2, 4))], bf16=True, opts={"grad2": 1}),
    _loss("bf16 V2000 L150", 2, 2000, 150, [(3, G1, (2, 3))], bf16=True),
]


def _proj_rows(tag, B, T, V, L, K, bf16, ctas, walk, entries):
    kern = {
        "proj_fwd": [(3, None, walk)],
        "proj_fwd_serial": [(3, None, walk)],
        "proj_loss_grad": [(4, G1, walk)],
        "proj_recompute": [(4, None, walk), (1, "any", None)],
        "proj_decode": [(4, None, walk)],
        "proj_decode_serial": [(4, None, walk)],
    }
    out = []
    for e in entries:
        opts = {"proj_overlap": 0} if e.endswith("_serial") else {}
        out.append(Row("%s %s" % (tag, e), e.replace("_serial", ""), B, T, V, L, kern[e], opts=opts, bf16=bf16, K=K,
                       ctas=ctas))
    return out


ALL_PROJ = ("proj_fwd", "proj_fwd_serial", "proj_loss_grad", "proj_recompute", "proj_decode", "proj_decode_serial")
PROJ_ROWS = (_proj_rows("V300 K64 fp32 ctas2", 3, 150, 300, 12, 64, False, 2, (1, 1), ALL_PROJ)
             + _proj_rows("V2000 K512 bf16 ctas1", 3, 200, 2000, 40, 512, True, 1, (2, 1), ALL_PROJ)
             + _proj_rows("V2000 K64 fp32 ctas1", 2, 150, 2000, 12, 64, False, 1, (1, 1), ("proj_loss_grad", "proj_recompute"))
             + _proj_rows("V300 K512 bf16 ctas2", 2, 150, 300, 12, 512, True, 2, (1, 1), ("proj_fwd", "proj_decode")))


def _other_row(row):
    """A different problem for the same buffer: a larger Lmax, the other vocabulary class, its own stamp."""
    V = 300 if row.V <= 64 else 46
    return Row("other", "loss_grad", row.B + 1, _T(row.L + 20, row.T + 16), V, row.L + 20, None)


# ---- inputs -------------------------------------------------------------------------------------------------------------
def _seed(name, k=0):
    return (sum(ord(c) * (i + 1) for i, c in enumerate(name)) + 7919 * k) % (2 ** 31)


def _pad_hostile(d, pred_or_hidden):
    """Frames t >= T_b get NaN, +-inf and +-3e38 in turn, label slots past L_b get 1e10, -7 and NaN in turn."""
    x = pred_or_hidden.copy()
    lab = d["label"].copy()
    Tb, Lb = d["pred_lengths"].astype(int), d["label_lengths"].astype(int)
    for b in range(x.shape[0]):
        for t in range(Tb[b], x.shape[1]):
            x[b, t] = PAD_LOGITS[(t + b) % len(PAD_LOGITS)]
        for j in range(Lb[b], lab.shape[1]):
            lab[b, j] = PAD_LABELS[(j + b) % len(PAD_LABELS)]
    return x, lab


def _inputs(dev, row, k=0, hostile=False):
    """Device inputs of one problem of ``row`` (seed k), and the host arrays the oracle needs."""
    B, T, V, L = row.B, row.T, row.V, row.L
    d = make_batch(B, T, V, L, seed=_seed(row.name, k))
    head = np.linspace(0.5, 1.5, B)
    inp = {"head": torch.tensor(head, device=dev, dtype=torch.float32), "np": d, "head_np": head}
    if row.proj:
        h, w, bv = _weights(B, T, row.K, V, seed=_seed(row.name, k) + 1, bf16=row.bf16)
        inp["logits64"] = _logits64(h, w, bv)
        lab = d["label"]
        if hostile:
            h, lab = _pad_hostile(d, h)
        th, tw = torch.tensor(h, device=dev), torch.tensor(w, device=dev)
        if row.bf16:
            th, tw = th.bfloat16(), tw.bfloat16()
        inp.update(hidden=th, weight=tw, bias=torch.tensor(bv, device=dev))
    else:
        x, lab = _pad_hostile(d, d["pred"]) if hostile else (d["pred"], d["label"])
        pred = torch.tensor(x, device=dev)
        if row.bf16:
            pred = pred.bfloat16()
            d = dict(d, pred=torch.tensor(d["pred"]).bfloat16().float().numpy())    # what the oracle sees: the bf16 values
            inp["np"] = d
        inp["pred"] = pred
    inp["label"] = torch.tensor(lab, device=dev)
    inp["pl"] = torch.tensor(d["pred_lengths"], device=dev)
    inp["ll"] = torch.tensor(d["label_lengths"], device=dev)
    return inp


def _outputs(dev, row, inp):
    B, T, V = row.B, row.T, row.V
    out = {"loss": torch.full((B,), NAN, device=dev),
           "status": torch.full((B,), -1, dtype=torch.int32, device=dev),
           "loss_sum": torch.zeros((1,), dtype=torch.float64, device=dev)}
    if row.need_grad:
        dt = inp["pred"].dtype if not row.proj else torch.float32
        out["grad"] = torch.full((B, T, V), NAN, device=dev, dtype=dt)
    if row.entry == "proj_decode":
        out["tokens"] = torch.full((B, T), -1, dtype=torch.int32, device=dev)
        out["lengths"] = torch.full((B,), -1, dtype=torch.int32, device=dev)
    return out


# ---- one row's C calls ----------------------------------------------------------------------------------------------------
def _enqueue(dev, row, inp, out, ws, nbytes):
    """Enqueues the row's C calls on the current stream into ``ws`` (``nbytes`` of it), without a synchronisation.
    Returns what each call launched: [(launches, gradient kernel, walker configuration)]."""
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _Call, _stream_ptr
    from gluon_e2e_asr_b200.proj import _MetaLogits, _proj_struct
    l = _lib.load()
    s = _stream_ptr(dev)
    kern = []

    def took(rc):
        _lib.check(rc)
        kern.append((_lib.last_launch_count(), _lib.last_grad_kernel(), _lib.last_walk_config()))

    if not row.proj:
        call = _Call(inp["pred"], inp["label"], inp["pl"], inp["ll"], False, True, False)
        if row.entry == "loss_grad":
            p = call.problem(out["loss"], out["grad"], inp["head"], out["loss_sum"], out["status"])
            took(l.ctcb_loss_grad_typed(ctypes.byref(p), call.ldt, ws, nbytes, s))
        elif row.entry == "forward":
            p = call.problem(out["loss"], None, None, out["loss_sum"], out["status"])
            took(l.ctcb_forward_typed(ctypes.byref(p), call.ldt, 0, ws, nbytes, s))
        else:                                                        # split
            p = call.problem(out["loss"], None, None, out["loss_sum"], out["status"])
            took(l.ctcb_forward_typed(ctypes.byref(p), call.ldt, 1, ws, nbytes, s))
            out["_scratch"] = torch.empty_like(out["loss"])
            p2 = call.problem(out["_scratch"], out["grad"], inp["head"])
            took(l.ctcb_backward_typed(ctypes.byref(p2), call.ldt, ws, nbytes, s))
        return kern
    B, T, V = row.B, row.T, row.V
    pj = _proj_struct(inp["hidden"], inp["weight"], inp["bias"])
    if row.entry == "proj_loss_grad":
        out["_logits"] = torch.full((B, T, V), NAN, device=dev)
        call = _Call(out["_logits"], inp["label"], inp["pl"], inp["ll"], False, True, False)
        p = call.problem(out["loss"], out["grad"], inp["head"], out["loss_sum"], out["status"])
        took(l.ctcb_proj_loss_grad(ctypes.byref(pj), ctypes.byref(p), ws, nbytes, s))
        return kern
    call = _Call(_MetaLogits(torch.empty((B, T, V), device="meta"), dev), inp["label"], inp["pl"], inp["ll"], False, True,
                 False)
    p = call.problem(out["loss"], None, None, out["loss_sum"], out["status"])
    p.logits = None
    if row.entry == "proj_fwd":
        took(l.ctcb_proj_forward(ctypes.byref(pj), ctypes.byref(p), 0, ws, nbytes, s))
    elif row.entry == "proj_decode":
        took(l.ctcb_proj_forward_decode(ctypes.byref(pj), ctypes.byref(p), 0, -1, out["tokens"].data_ptr(),
                                        out["lengths"].data_ptr(), ws, nbytes, s))
    else:                                                            # proj_recompute
        took(l.ctcb_proj_forward(ctypes.byref(pj), ctypes.byref(p), 1, ws, nbytes, s))
        out["_scratch"] = torch.empty_like(out["loss"])
        p2 = call.problem(out["_scratch"], out["grad"], inp["head"])
        p2.logits = None
        took(l.ctcb_proj_backward(ctypes.byref(pj), ctypes.byref(p2), ws, nbytes, s))
    return kern


def _check_kernels(row, kern):
    assert len(kern) == len(row.kern), row.name
    for i, ((n, gk, walk), (en, egk, ewalk)) in enumerate(zip(kern, row.kern)):
        assert n == en, "%s call %d: %d launches, expected %d" % (row.name, i, n, en)
        if egk != "any":
            assert gk == egk, "%s call %d: gradient kernel %s, expected %s" % (row.name, i, gk, egk)
        if ewalk is not None:
            assert walk == ewalk, "%s call %d: walker configuration %s, expected %s" % (row.name, i, walk, ewalk)


def _automatic(row):
    """The row's forced options set back to automatic (-1)."""
    return {k: -1 for k in row.opts}


def _fill(dev, ws, state, seed):
    if state == "zero":
        ws.zero_()
    elif state == "ff":
        ws.fill_(0xFF)
    elif state == "7f":
        ws.fill_(0x7F)
    elif state == "random":
        g = torch.Generator(device=dev).manual_seed(seed)
        ws.copy_(torch.randint(0, 256, ws.shape, generator=g, device=dev, dtype=torch.int16).to(torch.uint8))
    else:
        ws.fill_(0xA5)


def _run(dev, row, inp, state="zero", nbytes=None, dirty=None):
    """The row on a fresh workspace of ``nbytes`` in ``state``; ``dirty``: (row, inputs, options) enqueued into it first,
    under its own options."""
    from gluon_e2e_asr_b200 import _lib
    nbytes = nbytes or row.ws_bytes()
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    _fill(dev, ws, state, _seed(row.name, 99))
    if dirty is not None:
        drow, dinp, dopts = dirty
        with _lib.options(**dopts):
            _enqueue(dev, drow, dinp, _outputs(dev, drow, dinp), ws.data_ptr(), nbytes)    # no synchronisation in between
    out = _outputs(dev, row, inp)
    kern = _enqueue(dev, row, inp, out, ws.data_ptr(), nbytes)
    torch.cuda.synchronize()
    return out, kern


def _bits(t):
    if t.dtype == torch.bfloat16:
        return t.contiguous().view(torch.int16)
    if t.dtype == torch.float32:
        return t.contiguous().view(torch.int32)
    return t


def _same_bits(ref, got, what):
    for k, a in ref.items():
        if k.startswith("_"):
            continue
        b = got[k]
        if k == "loss_sum":
            x, y = float(a.item()), float(b.item())
            assert abs(x - y) <= 1e-12 * abs(x), "%s: loss_sum %r against %r" % (what, y, x)
            continue
        if not torch.equal(_bits(a), _bits(b)):
            diff = (_bits(a) != _bits(b)).nonzero()
            raise AssertionError("%s: %s differs in %d elements, first at %s (%r against %r)"
                                 % (what, k, diff.shape[0], tuple(diff[0].tolist()), b[tuple(diff[0].tolist())].item(),
                                    a[tuple(diff[0].tolist())].item()))


def _tokens_ref(dev, row, inp):
    """The decode's reference: ctcb_proj_loss_grad stores the logits the same tiles form; the numpy greedy decode of them
    (ties: lowest index)."""
    from gluon_e2e_asr_b200 import _lib
    lrow = Row("tokens", "proj_loss_grad", row.B, row.T, row.V, row.L, None, bf16=row.bf16, K=row.K, ctas=row.ctas)
    with _lib.options(**dict(_automatic(row), **lrow.opts)):
        out, _ = _run(dev, lrow, inp)
    return O.greedy_decode(out["_logits"].cpu().numpy(), inp["np"]["pred_lengths"], 0)


def _against_oracle(dev, row, inp, out):
    """The zero run meets the project's bar against the fp64 C oracle (tokens: exactly)."""
    d, head = inp["np"], inp["head_np"]
    if row.proj:
        lo, go, _ = _oracle(inp["logits64"], d["label"], d["pred_lengths"], d["label_lengths"], head, 0)
        st = O.param_layer(d["label"], d["pred_lengths"], d["label_lengths"], row.T, row.V, "first")[3]
    else:
        lo, go, st, _ = _expect(d, False, head)
    np.testing.assert_allclose(out["loss"].cpu().numpy(), lo, rtol=RTOL, atol=ATOL, err_msg=row.name + " loss")
    np.testing.assert_array_equal(out["status"].cpu().numpy(), st, err_msg=row.name + " status")
    np.testing.assert_allclose(out["loss_sum"].item(), lo.sum(), rtol=RTOL, err_msg=row.name + " loss_sum")
    if "grad" in out:
        g = out["grad"].float().cpu().numpy()
        rtol = GRAD_RTOL_BF16 if row.bf16 and not row.proj else RTOL
        np.testing.assert_allclose(g, go, rtol=rtol, atol=ATOL, err_msg=row.name + " grad")
    if "tokens" in out:
        ref = _tokens_ref(dev, row, inp)
        t, n = out["tokens"].cpu().numpy(), out["lengths"].cpu().numpy()
        for b, seq in enumerate(ref):
            assert n[b] == len(seq) and list(t[b, :n[b]]) == list(seq), "%s tokens of utterance %d" % (row.name, b)
            assert (t[b, n[b]:] == 0).all(), row.name


def _padded_rows_zero(row, inp, out, what):
    if "grad" not in out:
        return
    g = out["grad"].float().cpu().numpy()
    for b, n in enumerate(inp["np"]["pred_lengths"].astype(int)):
        assert (g[b, n:] == 0).all(), "%s: padded gradient rows of utterance %d are not 0" % (what, b)


# ---- A + B + E: every row, every workspace state, hostile padding ------------------------------------------------------------
@pytest.mark.parametrize("row", ROWS + PROJ_ROWS, ids=[r.name for r in ROWS + PROJ_ROWS])
def test_row_on_dirty_memory(dev, row):
    from gluon_e2e_asr_b200 import _lib
    other = _other_row(row)
    with _lib.options(**row.opts):
        inp = _inputs(dev, row)
        nbytes = max(row.ws_bytes(), other.ws_bytes())
        ref, kern = _run(dev, row, inp, "zero", nbytes)
        _check_kernels(row, kern)
        _against_oracle(dev, row, inp, ref)
        _padded_rows_zero(row, inp, ref, row.name)
        # the other problem runs under the automatic options, the same shape under the row's own
        dirt = {"other": (other, _inputs(dev, other), _automatic(row)), "same": (row, _inputs(dev, row, k=1), {})}
        for state in STATES[1:]:
            got, kern = _run(dev, row, inp, state, nbytes, dirt.get(state))
            _check_kernels(row, kern)
            _same_bits(ref, got, "%s, workspace %s" % (row.name, state))
        # E: hostile padded frames (hidden rows) and label slots, explicit lengths
        got, kern = _run(dev, row, _inputs(dev, row, hostile=True), "zero", nbytes)
        _check_kernels(row, kern)
        _same_bits(ref, got, "%s, hostile padding" % row.name)
        _padded_rows_zero(row, inp, got, row.name + " hostile padding")


# ---- C: one buffer for a bucketed loop ----------------------------------------------------------------------------------------
BUCKETS = [
    _loss("loop fused B3 L12", 3, 46, 12, None),
    _loss("loop fused B5 L100", 5, 46, 100, None),
    _loss("loop V300 B4 L30", 4, 300, 30, None),
    _loss("loop V2000 B2 L150", 2, 2000, 150, None),
    _loss("loop bf16 B3 L50", 3, 46, 50, None, bf16=True),
    _loss("loop forward V46 B6 L40", 6, 46, 40, None, entry="forward"),
    _loss("loop forward V300 B3 L20", 3, 300, 20, None, entry="forward"),
] + [Row("loop " + e, e, 3, 150, V, L, None, K=64) for e, V, L in
     (("proj_fwd", 300, 12), ("proj_loss_grad", 300, 20), ("proj_recompute", 2000, 12), ("proj_decode", 300, 16))]


def test_one_buffer_for_a_bucketed_loop(dev):
    """Eleven problems of mixed B, T, Lmax and V in {46, 300, 2000}, device loss, forward-only and projection entries,
    enqueued back to back into ONE workspace sized for the largest, with no synchronisation, then again in reverse order:
    every result has the bits of the same problem run alone on a fresh buffer."""
    inps = [_inputs(dev, r) for r in BUCKETS]
    alone = [_run(dev, r, i)[0] for r, i in zip(BUCKETS, inps)]
    nbytes = max(r.ws_bytes() for r in BUCKETS)
    ws = torch.full((nbytes,), 0xFF, dtype=torch.uint8, device=dev)
    for order in (range(len(BUCKETS)), reversed(range(len(BUCKETS)))):
        order = list(order)
        outs = {}
        for i in order:
            outs[i] = _outputs(dev, BUCKETS[i], inps[i])
            _enqueue(dev, BUCKETS[i], inps[i], outs[i], ws.data_ptr(), nbytes)
        torch.cuda.synchronize()
        for i in order:
            _same_bits(alone[i], outs[i], "%s in the shared buffer (order %s)" % (BUCKETS[i].name, order[:2]))


# ---- D: graph replay on a recycled workspace --------------------------------------------------------------------------------
def test_graph_replays_on_an_overwritten_workspace(dev):
    """A captured training step (ctc_loss_and_grad, pointer hand-off, cfg2's shape) and a captured projection loss
    evaluation: between replays their workspaces are filled with 0xFF and with another problem's call (what graphs that
    share a memory pool do to each other).  Every replay gives the bits of the eager call.  (A build whose fused walkers
    do not reset their progress words at entry can fail here, when the gradient CTAs trust the previous replay's words
    and get ahead of the walkers: it did in one of two runs.)"""
    from gluon_e2e_asr_b200 import _lib, ctc_loss_and_grad, ops
    from gluon_e2e_asr_b200.proj import _MetaLogits, _proj_struct
    B, T, V, L = 32, 500, 46, 120
    d = make_batch(B, T, V, L, seed=41)
    args = tuple(torch.tensor(d[k], device=dev) for k in ("pred", "label", "pred_lengths", "label_lengths"))
    l0, g0 = (t.clone() for t in ctc_loss_and_grad(*args))
    loss, grad = torch.empty_like(l0), torch.empty_like(g0)
    s = torch.cuda.Stream(dev)
    other = Row("graph other", "loss_grad", 8, 200, 300, 30, None)
    oinp = _inputs(dev, other)
    # the projection problem, on a workspace this test owns (large enough for the other problem too)
    prow = Row("graph proj", "proj_fwd", 4, 150, 300, 12, None, K=64)
    pinp = _inputs(dev, prow)
    pnbytes = max(prow.ws_bytes(), other.ws_bytes())
    pws = torch.zeros((pnbytes,), dtype=torch.uint8, device=dev)
    pref, _ = _run(dev, prow, pinp, "zero", pnbytes)
    pout = _outputs(dev, prow, pinp)
    with torch.cuda.stream(s):
        ctc_loss_and_grad(*args, out_loss=loss, out_grad=grad, handoff="pointer")     # warms the workspace cache
        _enqueue(dev, prow, pinp, pout, pws.data_ptr(), pnbytes)
        torch.cuda.synchronize()
        ws = ops._ws_cache[(dev.index, s.cuda_stream, T, B, V, L)]
        g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(g1, stream=s):
            ctc_loss_and_grad(*args, out_loss=loss, out_grad=grad, handoff="pointer")
        with torch.cuda.graph(g2, stream=s):
            _enqueue(dev, prow, pinp, pout, pws.data_ptr(), pnbytes)
    assert other.ws_bytes() <= ws.numel()
    for how in ("replay", "0xFF", "other problem", "0xFF"):
        with torch.cuda.stream(s):
            for buf, n in ((ws, ws.numel()), (pws, pnbytes)):
                if how == "0xFF":
                    buf.fill_(0xFF)
                elif how == "other problem":
                    _enqueue(dev, other, oinp, _outputs(dev, other, oinp), buf.data_ptr(), n)
            loss.fill_(NAN); grad.fill_(NAN)
            for k in ("loss", "status"):
                pout[k].fill_(NAN if k == "loss" else -1)
            pout["loss_sum"].zero_()
            g1.replay()
            g2.replay()
        torch.cuda.synchronize()
        assert torch.equal(_bits(loss), _bits(l0)) and torch.equal(_bits(grad), _bits(g0)), "training step after " + how
        _same_bits(pref, pout, "projection evaluation after " + how)
