"""GPU tests of the loss evaluation with the greedy decode on logits (ctcb_forward_decode_typed, ops.ctc_eval,
CtcLoss.evaluate).

The references are the two calls it replaces, on the same logits and under the same options: ctcb_forward_typed with
keep_for_backward = 0 (losses and status words bit for bit, the same walker configuration) and ctcb_greedy_decode_typed
(the whole (B, T) token tensor -- hypothesis and the zeros after it -- and the lengths, bit for bit).  better() is a
total order on the non-NaN {value, index} pairs and nothing is rounded, so any difference is a bug.  Every decoding call
runs on outputs pre-filled with garbage and on a workspace that is not clean."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from tests.synth import CONFIGS, make_batch

pytestmark = pytest.mark.gpu

GARBAGE = 0x5EADBEEF


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _fill(ws, state, seed=0):
    if state == "zero":
        ws.zero_()
    elif state == "ff":
        ws.fill_(0xFF)
    else:
        g = torch.Generator(device=ws.device).manual_seed(seed)
        ws.copy_(torch.randint(0, 256, ws.shape, generator=g, device=ws.device, dtype=torch.int16).to(torch.uint8))


class Case:
    """One problem: logits x (a view in any layout), labels, lengths and how the C problem is formed."""

    def __init__(self, x, lab, pl=None, ll=None, ntc=True, tn=False, blank_last=False, unk=None, opts=None, packed=False):
        from gluon_e2e_asr_b200.ops import _Call
        self.x, self.lab, self.pl, self.ll, self.unk = x, lab, pl, ll, unk
        self.ntc, self.blank_last, self.opts, self.packed = ntc, blank_last, dict(opts or {}), packed
        self.call = _Call(x, lab, pl, ll, blank_last, ntc, tn)
        self.blank = self.call.V - 1 if blank_last else 0
        if packed:
            # utterance b's valid frames back to back (ctcb_problem_t::logits_row_offsets)
            T, V = self.call.T, self.call.V
            n = [max(0, min(T, int(v))) for v in pl.cpu().numpy()]
            rows = [x[b, :n[b]] for b in range(self.call.B)]
            self.xp = torch.cat(rows + [x.new_zeros((1, V))]).contiguous()
            self.offs = torch.tensor(np.concatenate([[0], np.cumsum(n)[:-1]]) * V, dtype=torch.int64, device=x.device)

    def problem(self, loss, status):
        p = self.call.problem(loss, status=status)
        if self.packed:
            p.logits, p.logits_stride_t, p.logits_stride_b = self.xp.data_ptr(), self.call.V, 0
            p.logits_row_offsets = self.offs.data_ptr()
        return p

    def fused(self):
        return self.call.V <= 64 and self.opts.get("fused", -1) != 0


def _reference(c, ws):
    """ctcb_forward_typed(keep_for_backward = 0) and ctcb_greedy_decode_typed: the two calls the entry replaces."""
    from gluon_e2e_asr_b200 import _lib, greedy_decode
    from gluon_e2e_asr_b200.ops import _stream_ptr
    B = c.call.B
    loss = torch.full((B,), float("nan"), device=c.x.device)
    status = torch.full((B,), -1, dtype=torch.int32, device=c.x.device)
    p = c.problem(loss, status)
    _lib.check(_lib.load().ctcb_forward_typed(ctypes.byref(p), c.call.ldt, 0, ws.data_ptr(), ws.numel(), _stream_ptr(c.x.device)))
    launches, cfg = _lib.last_launch_count(), _lib.last_walk_config()
    toks, lens = greedy_decode(c.x, c.pl, c.blank, "NTC" if c.ntc else "TNC", c.unk)
    return dict(loss=loss, status=status, toks=toks, lens=lens, launches=launches, cfg=cfg)


def _decode(c, ws, out=None):
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _stream_ptr
    B, T = c.call.B, c.call.T
    dv = c.x.device
    out = out or dict(loss=torch.empty((B,), device=dv), status=torch.empty((B,), dtype=torch.int32, device=dv),
                      toks=torch.empty((B, T), dtype=torch.int32, device=dv), lens=torch.empty((B,), dtype=torch.int32, device=dv))
    out["loss"].fill_(float("nan")); out["status"].fill_(-1); out["toks"].fill_(GARBAGE); out["lens"].fill_(GARBAGE)
    p = c.problem(out["loss"], out["status"])
    _lib.check(_lib.load().ctcb_forward_decode_typed(ctypes.byref(p), c.call.ldt, -1 if c.unk is None else int(c.unk),
                                                     out["toks"].data_ptr(), out["lens"].data_ptr(), ws.data_ptr(),
                                                     ws.numel(), _stream_ptr(dv)))
    out["launches"], out["cfg"] = _lib.last_launch_count(), _lib.last_walk_config()
    return out


def _same(ref, got, what):
    torch.cuda.synchronize()
    for k in ("loss", "status", "toks", "lens"):
        a, b = _bits(ref[k]), _bits(got[k])
        if not torch.equal(a, b):
            bad = (a != b).nonzero()[:4].tolist()
            raise AssertionError("%s: %s differs at %s" % (what, k, bad))


def check(c, state="ff", seed=0, what=""):
    """The entry against the two-call path: bits, walker configuration, launch counts."""
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _alloc_ws
    with _lib.options(**c.opts):
        ws = _alloc_ws(c.call, False)
        _fill(ws, "zero")
        ref = _reference(c, ws)
        _fill(ws, state, seed)
        got = _decode(c, ws)
    what = what or "B=%d T=%d V=%d %s unk=%s opts=%s" % (c.call.B, c.call.T, c.call.V, c.x.dtype, c.unk, c.opts)
    _same(ref, got, what)
    assert got["cfg"] == ref["cfg"], what
    # V <= 64 fused: walkers, collapse; otherwise k_emit, walkers, collapse
    assert got["launches"] == (2 if c.fused() else 3) == ref["launches"] + 1, (what, got["launches"], ref["launches"])
    return ref, got


def _tensors(dev, d, dtype=torch.float32):
    x = torch.tensor(d["pred"], device=dev).to(dtype)
    return x, torch.tensor(d["label"], device=dev), torch.tensor(d["pred_lengths"], device=dev), torch.tensor(d["label_lengths"], device=dev)


def _ties(dev, B, T, V, seed, dtype):
    """Integer-valued logits in a narrow range: exact ties within a lane's columns, across lanes and vector loads."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randint(-2, 2, (B, T, V), generator=g).to(dtype).to(dev)


# ---- the reference's shapes ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg,dtype", [("cfg1", "f32"), ("cfg2", "f32"), ("cfg3", "f32"), ("cfg4", "f32"), ("cfg5", "f32"),
                                       ("cfg2", "bf16"), ("cfg3", "bf16")])
def test_reference_shapes(dev, cfg, dtype):
    """cfg1-cfg5 (cfg5, B = 1024: one walker per utterance, no meeting in the middle), unk unset / mid-vocabulary / the
    blank in turn, every workspace state."""
    B, T, V, L = CONFIGS[cfg]
    k = int(cfg[-1])
    x, lab, pl, ll = _tensors(dev, make_batch(B, T, V, L, seed=k), torch.bfloat16 if dtype == "bf16" else torch.float32)
    unk = (None, V // 2, 0)[k % 3]
    check(Case(x, lab, pl, ll, unk=unk), ("ff", "zero", "random")[k % 3], seed=k)


# ---- vocabularies, layouts, strides, ties ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("V", [46, 64, 65, 66, 300, 2000])
def test_vocabularies_layouts_and_ties(dev, V, dtype):
    """Integer-valued logits (exact ties everywhere) in NTC and TNC, as a column slice of a wider tensor (row stride !=
    V), from an offset base (VEC 1), V % 4 != 0 (VEC 1 / 2, register-resident k_emit), packed logits, blank_label="last"
    and each <unk> choice."""
    B, T, L = 6, 90, 20
    d = make_batch(B, T, V, L, seed=V)
    _, lab, pl, ll = _tensors(dev, d)
    pl[0] = T
    x = _ties(dev, B, T, V, V, dtype)
    check(Case(x, lab, pl, ll, unk=V // 3))
    check(Case(x.transpose(0, 1).contiguous().transpose(0, 1), lab, pl, ll, ntc=True, unk=0))    # (B,T) strides of TNC storage
    check(Case(x.transpose(0, 1).contiguous(), lab, pl, ll, ntc=False, unk=None))
    wide = _ties(dev, B, T, V + 5, V + 1, dtype)
    check(Case(wide[:, :, :V], lab, pl, ll, unk=V - 1))
    check(Case(wide[:, :, 1:V + 1], lab, pl, ll, unk=None))
    check(Case(x, lab, pl, ll, unk=2, packed=True))
    lab_last = torch.where(lab == 0, torch.full_like(lab, -1), lab - 1)      # blank V - 1, labels 0..V-2, padding -1
    check(Case(x, lab_last, pl, ll, blank_last=True, unk=V - 1))
    check(Case(x, lab_last, pl, ll, blank_last=True, unk=None))


@pytest.mark.parametrize("opts", [dict(emit_staged=0), dict(fused=0), dict(meet_fwd=0), dict(meet_fwd=1), dict(walk_pdl=0)])
@pytest.mark.parametrize("V", [46, 2000])
def test_options(dev, V, opts):
    """Every route the options select: the staged emit off, k_emit for V <= 64 (fused=0), the walkers meeting in the
    middle forced off and on, the fused walkers without the programmatic launch."""
    B, T, L = 12, 160, 40
    x, lab, pl, ll = _tensors(dev, make_batch(B, T, V, L, seed=3))
    for unk in (None, 5):
        for dtype in (torch.float32, torch.bfloat16):
            check(Case(x.to(dtype), lab, pl, ll, unk=unk, opts=opts))


@pytest.mark.parametrize("pc", [(1, 1), (2, 1), (2, 2), (2, 3), (2, 4), (2, 5), (2, 6), (2, 8), (2, 12), (2, 16), (4, 16)])
def test_every_default_walker_configuration(dev, pc):
    """The configuration the label length picks, from (1, 1) to (4, 16), fused walkers with the decode in their
    producers; pinned through ctcb_last_walk_config."""
    P, NW = pc
    L = P * NW * 32 - 1
    B, V = 3, 46
    T = 2 * L + 24
    d = make_batch(B, T, V, L, seed=P * 100 + NW, full_lengths=True)
    x, lab, pl, ll = _tensors(dev, d)
    pl[1] = T - 7
    for dtype, unk in ((torch.float32, None), (torch.bfloat16, 3)):
        ref, got = check(Case(x.to(dtype), lab, pl, ll, unk=unk))
        assert got["cfg"] == (P, NW)


# ---- hostile rows and lengths --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("V", [46, 300])
def test_hostile_rows_and_lengths(dev, V):
    """Rows of all -inf, all NaN and mixed +-inf; infeasible utterances, T_b = 0, L = 0, lengths below 0 and above T,
    fractional lengths, in every length dtype."""
    B, T, L = 8, 64, 12
    d = make_batch(B, T, V, L, seed=17)
    x, lab, _, _ = _tensors(dev, d)
    x[0, 3] = float("-inf")
    x[1, 5] = float("nan")
    x[2, 7, ::2] = float("inf")
    x[2, 7, 1::2] = float("-inf")
    x[3, 9, V // 2] = float("nan")
    x[4, 2, 1] = float("inf")
    pls = [T, T, T, 3, 0, -5, T + 40, 40.7]          # utterance 3: 3 frames for 12 labels (infeasible)
    lls = [L, 0, L, L, L, L + 9, -2, 5.5]
    for dt in (torch.int32, torch.int64, torch.float32, torch.float64):
        pl = torch.tensor(pls, dtype=dt, device=dev)
        ll = torch.tensor(lls, dtype=dt, device=dev)
        for unk in (None, 1):
            for dtype in (torch.float32, torch.bfloat16):
                check(Case(x.to(dtype), lab, pl, ll, unk=unk))
    # every utterance infeasible (the CTAs return before their producers run) and without data_lengths
    x2, lab2 = x[:, :5].clone(), torch.ones((B, L), device=dev)
    check(Case(x2, lab2, None, None, unk=None))
    check(Case(x2, lab2, torch.tensor([5, 0, 2, 5, 1, 3, 4, 5], device=dev), None, unk=2))


# ---- memory state --------------------------------------------------------------------------------------------------------
def test_one_workspace_for_back_to_back_calls_of_different_shapes(dev):
    """Decoding calls of different shapes and routes enqueued back to back into one workspace sized for the largest,
    without synchronisation: every result has the bits of the same call run alone."""
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _alloc_ws
    cases = []
    for k, (B, T, V, L) in enumerate([(8, 200, 46, 50), (16, 120, 2000, 30), (4, 300, 65, 60), (32, 80, 46, 20), (6, 100, 300, 25)]):
        x, lab, pl, ll = _tensors(dev, make_batch(B, T, V, L, seed=50 + k))
        cases.append(Case(x, lab, pl, ll, unk=(None, 3)[k % 2]))
    alone = []
    for c in cases:
        ws = _alloc_ws(c.call, False)
        _fill(ws, "ff")
        alone.append({k: (v.clone() if torch.is_tensor(v) else v) for k, v in _decode(c, ws).items()})
    ws = torch.full((max(_alloc_ws(c.call, False).numel() for c in cases),), 0xA5, dtype=torch.uint8, device=dev)
    for order in (list(range(len(cases))), list(reversed(range(len(cases))))):
        outs = {i: _decode(cases[i], ws) for i in order}
        for i in order:
            _same(alone[i], outs[i], "case %d in the shared buffer" % i)
    assert _lib.last_launch_count() in (2, 3)


def test_graph_replays_on_an_overwritten_workspace(dev):
    """A captured decoding loss evaluation (cfg2's shape, fused walkers; and V = 300, k_emit): between replays the
    workspace is filled with 0xFF, random bytes and another problem's call.  Every replay gives the eager call's bits."""
    from gluon_e2e_asr_b200.ops import _alloc_ws
    s = torch.cuda.Stream(dev)
    for (B, T, V, L) in ((32, 500, 46, 120), (8, 200, 300, 40)):
        x, lab, pl, ll = _tensors(dev, make_batch(B, T, V, L, seed=V))
        c = Case(x, lab, pl, ll, unk=4)
        ws = _alloc_ws(c.call, False)
        _fill(ws, "zero")
        ref = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in _reference(c, ws).items()}
        xo, labo, plo, llo = _tensors(dev, make_batch(4, 100, V, 10, seed=1))
        other = Case(xo, labo, plo, llo)
        torch.cuda.synchronize()                    # the reference ran on the default stream, on the same workspace
        with torch.cuda.stream(s):
            out = _decode(c, ws)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                _decode(c, ws, out)
        for how in ("replay", "ff", "random", "other problem"):
            with torch.cuda.stream(s):
                if how == "other problem":
                    _decode(other, ws)
                elif how != "replay":
                    _fill(ws, how, 7)
                out["loss"].fill_(float("nan")); out["toks"].fill_(GARBAGE); out["lens"].fill_(GARBAGE); out["status"].fill_(-1)
                g.replay()
            _same(ref, out, "V=%d graph replay after %s" % (V, how))


# ---- the public surface --------------------------------------------------------------------------------------------------
def test_ctc_eval_block_wer_and_oracle(dev):
    """ops.ctc_eval / CtcLoss.evaluate against ctc_loss under no_grad and greedy_decode; the WER totals of edit_distance
    against the two-call path's; the loss against the fp64 oracle once; no autograd graph; fp16 refused."""
    from gluon_e2e_asr_b200 import CtcLoss, ctc_eval, ctc_loss, edit_distance, greedy_decode
    from oracle.ctc_oracle import CtcLossOracle
    B, T, V, L = CONFIGS["cfg2"]
    d = make_batch(B, T, V, L, seed=9)
    x, lab, pl, ll = _tensors(dev, d)
    x.requires_grad_(True)
    loss, toks, lens = ctc_eval(x, lab, pl, ll, unk=7)
    assert not loss.requires_grad and loss.grad_fn is None
    with torch.no_grad():
        ref = ctc_loss(x.transpose(0, 1), lab, pl, ll, use_data_lengths=True, use_label_lengths=True)
    rt, rn = greedy_decode(x, pl, 0, unk=7)
    assert torch.equal(_bits(loss), _bits(ref)) and torch.equal(toks, rt) and torch.equal(lens, rn)
    lo, _, _ = CtcLossOracle("NTC", "NT")(d["pred"], d["label"], d["pred_lengths"], d["label_lengths"])
    np.testing.assert_allclose(loss.cpu().numpy(), lo, rtol=1e-4, atol=1e-5)
    # the validation loop of the reference with the block: loss, hypotheses, WER
    ref_tok = lab.to(torch.int32).contiguous()
    ref_len = ll.to(torch.int32)
    tot_a = torch.zeros(2, dtype=torch.int64, device=dev)
    tot_b = torch.zeros(2, dtype=torch.int64, device=dev)
    block = CtcLoss(layout="TNC", label_layout="NT", weight=0.5)
    xt = x.detach().transpose(0, 1)
    bl, bt, bn = block.evaluate(xt, lab, pl, ll)
    edit_distance(ref_tok, ref_len, bt, bn, totals=tot_a)
    with torch.no_grad():
        rl = block(xt, lab, pl, ll)
    rt2, rn2 = greedy_decode(xt, pl, 0, layout="TNC")
    edit_distance(ref_tok, ref_len, rt2, rn2, totals=tot_b)
    assert torch.equal(_bits(bl), _bits(rl)) and torch.equal(bt, rt2) and torch.equal(bn, rn2)
    assert torch.equal(tot_a, tot_b) and int(tot_a[1]) == int(ll.sum())
    with pytest.raises(TypeError) as e:
        ctc_eval(x.detach().half(), lab, pl, ll)
    assert "float16" in str(e.value)
