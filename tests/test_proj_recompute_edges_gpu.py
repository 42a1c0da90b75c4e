"""The recomputing training path of the fused projection (ctcb_proj_forward with keep_for_backward and no logits buffer,
then ctcb_proj_backward) at the edges where its two kernels can go wrong without the clean-input tests noticing:

  * hostile labels and lengths (tests/synth.py hostile_batch): k_proj_emit<..., kProjGrad> clamps labels and sorts the
    lattice columns by symbol itself, and subtracts a repeated symbol's occupancy once per lattice column;
  * every default walker configuration at the top of its range: k_proj_occ indexes the history by 32 P NW state pairs;
  * utterances with no frames to spare, where beta' is exactly zero on most states of the late frames;
  * G as a TNC buffer or as a view into a wider buffer (TMA tile stores and coalesced row stores), hidden as a TNC view,
    labels in TN layout;
  * random shapes, the emission floor, two graphs alive at once, and the single-CTA shared-memory limit.

References are fp64: the C oracle (oracle/ctc_ref) on the fp64 product of tf32-exact (or bfloat16) operands, after
oracle.ctc_oracle.param_layer's clamping where the inputs are hostile; and ctcb_proj_loss_grad (logits stored, k_grad) on
the same operands, whose losses must be bit-identical and whose G must agree to G_VS_LOGITS_PATH * max|head|.  Every G
buffer starts NaN-poisoned.  Helpers are copies of test_proj_recompute_gpu.py's and test_param_layer_gpu.py's."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import ctc_oracle as O
from oracle import ctc_ref
from tests.synth import hostile_batch, make_batch

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-4, 1e-5
# G against ctcb_proj_loss_grad's: the same softmax arithmetic, occupancies from the same 20-bit high words of the history
# normalised by two normalisers that agree to 2^-20 (test_proj_recompute_gpu.py)
G_VS_LOGITS_PATH = 4e-6
NAN = float("nan")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _tf32(x):
    return (np.ascontiguousarray(x, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def _bf16(x):
    return torch.tensor(np.ascontiguousarray(x, np.float32)).bfloat16().float().numpy()


def _weights(B, T, K, V, seed, bf16=False, bias=True):
    """hidden (B,T,K), weight (V,K), bias (V,) or None, exact in the operand type the kernel multiplies."""
    rng = np.random.Generator(np.random.PCG64(seed))
    h = rng.standard_normal((B, T, K)).astype(np.float32)
    w = (rng.standard_normal((V, K)) / np.sqrt(K)).astype(np.float32)
    bv = (rng.standard_normal((V,)) * 0.5).astype(np.float32) if bias else None
    rnd = _bf16 if bf16 else _tf32
    return rnd(h), rnd(w), bv


def _logits64(h, w, bv):
    x = h.astype(np.float64) @ w.astype(np.float64).T
    return x + bv.astype(np.float64) if bv is not None else x


def _operands(dev, h, w, bv, bf16=False):
    th, tw = torch.tensor(h, device=dev), torch.tensor(w, device=dev)
    if bf16:
        th, tw = th.bfloat16(), tw.bfloat16()
    return th, tw, (torch.tensor(bv, device=dev) if bv is not None else None)


def _dev_labels(dev, d):
    return tuple(None if d[k] is None else torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))


def _recompute(dev, ops, lab, pl, ll, head, blank_last=False, tn=False, G=None, status=False):
    """ctcb_proj_forward(keep=1, logits NULL) + ctcb_proj_backward through the C ABI.  ``G``: the (B,T,V) output view
    (default: a compact NaN-poisoned buffer).  Returns (loss, G, status or None, walker configuration (P, NW))."""
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _Call, _alloc_ws, _stream_ptr
    from gluon_e2e_asr_b200.proj import _MetaLogits, _proj_struct
    th, tw, tb = ops
    B, T, V = th.shape[0], th.shape[1], tw.shape[0]
    l = _lib.load()
    pj = _proj_struct(th, tw, tb)
    call = _Call(_MetaLogits(torch.empty((B, T, V), device="meta"), dev), lab, pl, ll, blank_last, True, tn)
    ws = _alloc_ws(call, True)
    loss = torch.full((B,), NAN, device=dev)
    st = torch.full((B,), -1, dtype=torch.int32, device=dev) if status else None
    p = call.problem(loss, status=st)
    p.logits = None
    _lib.check(l.ctcb_proj_forward(ctypes.byref(pj), ctypes.byref(p), 1, ws.data_ptr(), ws.numel(), _stream_ptr(dev)))
    assert _lib.last_launch_count() == 4          # k_proj_emit, metadata, k_walk, k_proj_occ
    walk = _lib.last_walk_config()
    if G is None:
        G = torch.full((B, T, V), NAN, device=dev)
    p2 = call.problem(torch.empty((B,), device=dev), grad=G, head=torch.tensor(head, device=dev, dtype=torch.float32))
    p2.logits = None
    _lib.check(l.ctcb_proj_backward(ctypes.byref(pj), ctypes.byref(p2), ws.data_ptr(), ws.numel(), _stream_ptr(dev)))
    assert _lib.last_launch_count() == 1
    torch.cuda.synchronize()
    return loss, G, st, walk


def _logits_path(dev, ops, lab, pl, ll, head, blank_last=False, status=False):
    """ctcb_proj_loss_grad on the same operands (the logits stored, k_grad): (loss, G, status or None)."""
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _Call, _alloc_ws, _stream_ptr
    from gluon_e2e_asr_b200.proj import _proj_struct
    th, tw, tb = ops
    B, T, V = th.shape[0], th.shape[1], tw.shape[0]
    logits = torch.full((B, T, V), NAN, device=dev)
    G = torch.full_like(logits, NAN)
    loss = torch.full((B,), NAN, device=dev)
    st = torch.full((B,), -1, dtype=torch.int32, device=dev) if status else None
    call = _Call(logits, lab, pl, ll, blank_last, True, False)
    ws = _alloc_ws(call, True)
    p = call.problem(loss, G, torch.tensor(head, device=dev, dtype=torch.float32), status=st)
    _lib.check(_lib.load().ctcb_proj_loss_grad(ctypes.byref(_proj_struct(th, tw, tb)), ctypes.byref(p), ws.data_ptr(),
                                               ws.numel(), _stream_ptr(dev)))
    torch.cuda.synchronize()
    return loss, G, st


def _np(t):
    return None if t is None else t.cpu().numpy()


def _against_logits_path(loss_c, G_c, loss_r, G_r, head, what):
    """(d): losses bit-identical, G finite and within G_VS_LOGITS_PATH * max|head| of the logits path's."""
    np.testing.assert_array_equal(loss_c, loss_r, err_msg=what + ": losses of ctcb_proj_loss_grad")
    assert np.isfinite(G_c).all(), what + ": NaN / inf left in G"
    assert np.isfinite(G_r).all(), what + ": NaN / inf left in the logits path's G"
    err = np.abs(G_c - G_r).max()
    assert err <= G_VS_LOGITS_PATH * np.max(head), "%s: |G - G_logits| = %.3e" % (what, err)


def _oracle(logits64, lab, Tb, Lb, head, blank):
    lo, G, feas = ctc_ref.ctc_ref(logits64, lab, Tb, Lb, blank=blank, head_grad=head, layout="NTC", dtype=np.float64)
    for b in range(G.shape[0]):                      # padded frames and infeasible utterances: exact zeros
        G[b, int(Tb[b]):] = 0.0
        if not feas[b]:
            G[b] = 0.0
    return lo, G, feas


# ---- 1. hostile labels and lengths --------------------------------------------------------------------------------------
HOSTILE = [
    # V, blank last, label / length dtype, rows, bf16 operands, proj_ctas
    (V, bl, dt, 1, False, 2) for V in (300, 600) for bl in (False, True) for dt in ("f32", "i64")
] + [
    (300, False, "f32", 17, False, 2),    # B = 306 > 296: the walkers are not all resident, the logits path runs serially
    (600, True, "f32", 1, True, 2),       # bfloat16 operands
    (300, True, "i64", 1, False, 1),      # single CTAs
]


@pytest.mark.parametrize("V,blank_last,dt,rows,bf16,ctas", HOSTILE,
                         ids=["V%d-%s-%s-rows%d%s-ctas%d" % (c[0], "last" if c[1] else "first", c[2], c[3],
                                                           "-bf16" if c[4] else "", c[5]) for c in HOSTILE])
def test_hostile_labels_and_lengths(dev, V, blank_last, dt, rows, bf16, ctas):
    """hostile_batch through the recomputing path, lengths given and inferred: (a) loss and G against the fp64 oracle of
    the clamped inputs, infeasible rows exactly 0; (b) the status word equals param_layer's; (c) the same bits as the batch
    clamped by hand (status bits 2 and 4 aside); (d) losses bit-identical to ctcb_proj_loss_grad's, G within its bound.
    Rows 15 and 16 clamp two labels >= V to one symbol (a repeat, which with blank 'last' is also the blank's column);
    the label columns of the forward go through the shared-memory stash (no logits store)."""
    from gluon_e2e_asr_b200 import _lib
    T, K, Lmax = 150, 64, 12
    blank = V - 1 if blank_last else 0
    bl = "last" if blank_last else "first"
    with _lib.options(proj_ctas=ctas):
        for inferred in (False, True):
            d = hostile_batch(T, V, Lmax, blank_last=blank_last, label_dtype=dt, length_dtype=dt, inferred=inferred,
                              seed=V + rows + 3, rows=rows * 18 // 8 if inferred else rows)
            B = d["label"].shape[0]
            h, w, bv = _weights(B, T, K, V, seed=V + 11, bf16=bf16)
            head = np.linspace(0.5, 1.5, B)
            what = "V=%d blank %s %s inferred=%s" % (V, bl, dt, inferred)
            Tb, Lb, lab, st = O.param_layer(d["label"], d["pred_lengths"], d["label_lengths"], T, V, bl)
            lo, go, feas = _oracle(_logits64(h, w, bv), lab, Tb, Lb, head, blank)
            np.testing.assert_array_equal(feas, (st & 1) == 0)
            infeasible = (st & 1) != 0
            assert infeasible.any(), what
            ops = _operands(dev, h, w, bv, bf16)
            loss, G, status, _ = _recompute(dev, ops, *_dev_labels(dev, d), head, blank_last, status=True)
            l_c, G_c, s_c = _np(loss), _np(G), _np(status)
            # (a)
            np.testing.assert_allclose(l_c, lo, rtol=RTOL, atol=ATOL, err_msg=what + " loss")
            np.testing.assert_allclose(G_c, go, rtol=RTOL, atol=ATOL, err_msg=what + " G")
            assert (l_c[infeasible] == 0).all() and (G_c[infeasible] == 0).all(), what
            # (b)
            np.testing.assert_array_equal(s_c, st, err_msg=what + " status word")
            # (c) the same batch clamped by hand
            dc = dict(label=lab.astype(np.float32), pred_lengths=Tb.astype(np.float32), label_lengths=Lb.astype(np.float32))
            loss2, G2, status2, _ = _recompute(dev, ops, *_dev_labels(dev, dc), head, blank_last, status=True)
            assert torch.equal(loss, loss2), what + ": hostile and hand-clamped losses differ"
            assert torch.equal(G, G2), what + ": hostile and hand-clamped gradients differ"
            np.testing.assert_array_equal(s_c & ~6, _np(status2) & ~6, err_msg=what)
            # (d)
            loss_r, G_r, status_r = _logits_path(dev, ops, *_dev_labels(dev, d), head, blank_last, status=True)
            _against_logits_path(l_c, G_c, _np(loss_r), _np(G_r), head, what)
            np.testing.assert_array_equal(_np(status_r), st, err_msg=what + " status word of the logits path")


# ---- 2. every default walker configuration --------------------------------------------------------------------------------
# choose_walk (ctcb.cu) takes the first of these (P, NW) with 32 P NW >= Lmax + 1 state pairs:
#   (1,1) (2,1) (2,2) (2,3) (2,4) (2,5) (2,6) (2,8) (2,12) (2,16) (4,16)
# Each case sits at the top of its configuration's range, Lmax = 32 P NW - 1, so that the last state pair is a label state
# -- except (4,16): the walkers' emission ring of a gathered table (two stages of Lmax + 1 columns, 80 bytes each, within
# 200 KB) ends at Lmax = GATHERED_LMAX_MAX, and the projection only takes gathered tables (V > Lmax + 1).
WALKS = [(1, 1), (2, 1), (2, 2), (2, 3), (2, 4), (2, 5), (2, 6), (2, 8), (2, 12), (2, 16), (4, 16)]
GATHERED_LMAX_MAX = 1135


@pytest.mark.parametrize("P,NW", WALKS, ids=["P%d-NW%d" % w for w in WALKS])
def test_every_default_walker_configuration(dev, P, NW):
    """k_proj_occ (recomputing path) and k_grad (ctcb_proj_loss_grad) fed by every walker configuration, against the fp64
    C oracle.  One utterance has the full Lmax, the others are ragged; every utterance repeats a symbol twice (once at
    its start, once at its end).  V = max(65, Lmax + 2) + an odd offset: a gathered table whose last vocabulary tile is
    partial, G rows of V % 4 == 0 (TMA tile stores) and V % 4 == 2 (row stores) across the cases."""
    from gluon_e2e_asr_b200 import _lib
    Lmax = min(32 * P * NW - 1, GATHERED_LMAX_MAX)
    V = max(65, Lmax + 2) + (3 if NW % 2 == 0 else 5)
    T = 2 * Lmax + 41
    B, K = (3 if Lmax < 1000 else 2), 32
    rng = np.random.Generator(np.random.PCG64(Lmax))
    lab = rng.integers(1, V, (B, Lmax))
    Lb = np.concatenate([[Lmax], rng.integers(Lmax // 3, Lmax, B - 1)])
    Tb = np.full((B,), T)
    for b in range(B):
        lab[b, 1] = lab[b, 0]
        lab[b, Lb[b] - 1] = lab[b, Lb[b] - 2]
        lab[b, Lb[b]:] = 0
        reps = int((lab[b, 1:Lb[b]] == lab[b, :Lb[b] - 1]).sum())
        if b:
            Tb[b] = rng.integers(Lb[b] + reps, T)
    d = dict(label=lab.astype(np.float32), pred_lengths=Tb.astype(np.float32), label_lengths=Lb.astype(np.float32))
    h, w, bv = _weights(B, T, K, V, seed=Lmax + 1)
    head = np.linspace(0.5, 1.5, B)
    lo, go, feas = _oracle(_logits64(h, w, bv), lab, Tb, Lb, head, 0)
    assert feas.all()
    ops = _operands(dev, h, w, bv)
    labs = _dev_labels(dev, d)
    loss, G, _, walk = _recompute(dev, ops, *labs, head)
    assert walk == (P, NW), "walker configuration %s for Lmax=%d" % (walk, Lmax)
    l_c, G_c = _np(loss), _np(G)
    np.testing.assert_allclose(l_c, lo, rtol=RTOL, atol=ATOL, err_msg="recompute loss")
    np.testing.assert_allclose(G_c, go, rtol=RTOL, atol=ATOL, err_msg="recompute G")
    loss_r, G_r, _ = _logits_path(dev, ops, *labs, head)
    assert _lib.last_walk_config() == (P, NW)
    l_r, G_r = _np(loss_r), _np(G_r)
    np.testing.assert_allclose(l_r, lo, rtol=RTOL, atol=ATOL, err_msg="logits path loss")
    np.testing.assert_allclose(G_r, go, rtol=RTOL, atol=ATOL, err_msg="logits path G")
    _against_logits_path(l_c, G_c, l_r, G_r, head, "P=%d NW=%d" % (P, NW))


TIGHT = [(1023, 1028, 2), (511, 516, 4), (300, 305, 6), (120, 131, 8)]


@pytest.mark.parametrize("Lmax,V,B", TIGHT, ids=["L%d" % c[0] for c in TIGHT])
def test_tight_utterances(dev, Lmax, V, B):
    """Utterances with no or a few frames to spare (T_b = L_b + repeats + 0, 1, 3, 17): in their late frames most lattice
    states can no longer reach the end, so beta' is exactly 0 there while alpha is not.  k_proj_occ must count such a
    state as empty (as k_grad does): with the block's exponent shift applied, its alpha's high word can land on exponent
    2047, and inf * 0 left NaN occupancies, hence NaN entries of G.  Against the fp64 C oracle and the logits path."""
    rng = np.random.Generator(np.random.PCG64(Lmax + 7))
    lab = rng.integers(1, V, (B, Lmax))
    Lb = np.concatenate([[Lmax], rng.integers(Lmax // 2, Lmax + 1, B - 1)])
    Tb = np.zeros((B,), np.int64)
    for b in range(B):
        lab[b, Lb[b]:] = 0
        Tb[b] = Lb[b] + int((lab[b, 1:Lb[b]] == lab[b, :Lb[b] - 1]).sum()) + (0, 1, 3, 17)[b % 4]
    T = int(Tb.max())
    d = dict(label=lab.astype(np.float32), pred_lengths=Tb.astype(np.float32), label_lengths=Lb.astype(np.float32))
    h, w, bv = _weights(B, T, 32, V, seed=Lmax + 8)
    head = np.linspace(0.5, 1.5, B)
    lo, go, feas = _oracle(_logits64(h, w, bv), lab, Tb, Lb, head, 0)
    assert feas.all()
    ops = _operands(dev, h, w, bv)
    labs = _dev_labels(dev, d)
    loss, G, _, _ = _recompute(dev, ops, *labs, head)
    loss_r, G_r, _ = _logits_path(dev, ops, *labs, head)
    l_c, G_c = _np(loss), _np(G)
    assert np.isfinite(G_c).all(), "non-finite G in %d entries" % (~np.isfinite(G_c)).sum()
    np.testing.assert_allclose(l_c, lo, rtol=RTOL, atol=ATOL, err_msg="loss")
    np.testing.assert_allclose(G_c, go, rtol=RTOL, atol=ATOL, err_msg="G")
    _against_logits_path(l_c, G_c, _np(loss_r), _np(G_r), head, "tight Lmax=%d" % Lmax)


# ---- 4. output layouts and operand views ----------------------------------------------------------------------------------
def _layout_problem(dev, seed=81):
    B, T, K, V, L = 3, 150, 64, 300, 20           # T and V not multiples of 32: clipped tiles at both ends
    d = make_batch(B, T, V, L, seed=seed)
    h, w, bv = _weights(B, T, K, V, seed=seed + 1)
    return d, h, w, bv, np.linspace(0.5, 1.5, B)


def test_gradient_buffer_layouts(dev):
    """G as a TNC buffer, and as a view into a wider NaN-filled buffer whose row stride is a multiple of 4 (TMA tile
    stores: the clipped stores must write nothing past V or T) and one whose row stride is not (row stores): the same
    bits as the compact call, and nothing outside the view changes."""
    d, h, w, bv, head = _layout_problem(dev)
    B, T, V = h.shape[0], h.shape[1], w.shape[0]
    ops = _operands(dev, h, w, bv)
    labs = _dev_labels(dev, d)
    loss, G, _, _ = _recompute(dev, ops, *labs, head)
    assert torch.isfinite(G).all()
    G_tnc = torch.full((T, B, V), NAN, device=dev)
    loss2, _, _, _ = _recompute(dev, ops, *labs, head, G=G_tnc.transpose(0, 1))
    assert torch.equal(loss2, loss)
    assert torch.equal(G_tnc.transpose(0, 1), G), "TNC G"
    for pad in (4, 3):                             # row stride V + 4: TMA tile stores; V + 3: coalesced row stores
        buf = torch.full((B, T + 5, V + pad), NAN, device=dev)
        view = buf[:, 2:T + 2, :V]
        loss3, _, _, _ = _recompute(dev, ops, *labs, head, G=view)
        assert torch.equal(loss3, loss)
        assert torch.equal(view, G), "G view, row stride %d" % (V + pad)
        outside = torch.ones_like(buf, dtype=torch.bool)
        outside[:, 2:T + 2, :V] = False
        assert torch.isnan(buf[outside]).all(), "the call wrote outside the G view (row stride %d)" % (V + pad)


def test_hidden_as_a_tnc_view(dev):
    """hidden (T, B, K) transposed to (B, T, K): unit stride along K, so the projection reads it in place (no copy)."""
    d, h, w, bv, head = _layout_problem(dev, seed=83)
    ops = _operands(dev, h, w, bv)
    labs = _dev_labels(dev, d)
    loss, G, _, _ = _recompute(dev, ops, *labs, head)
    th_tnc = torch.tensor(np.ascontiguousarray(h.transpose(1, 0, 2)), device=dev).transpose(0, 1)
    assert th_tnc.stride(2) == 1 and not th_tnc.is_contiguous()
    loss2, G2, _, _ = _recompute(dev, (th_tnc,) + ops[1:], *labs, head)
    assert torch.equal(loss2, loss) and torch.equal(G2, G)


def test_tn_labels_through_proj_ctc_loss(dev):
    """label_layout="TN" (a (Lmax, B) label tensor) on the recomputing path: the same loss and parameter-gradient bits
    as the NT call."""
    from gluon_e2e_asr_b200 import proj_ctc_loss
    d, h, w, bv, head = _layout_problem(dev, seed=85)
    lab, pl, ll = _dev_labels(dev, d)
    out = []
    for tn in (False, True):
        th, tw, tb = (t.requires_grad_(True) for t in _operands(dev, h, w, bv))
        loss = proj_ctc_loss(th, tw, tb, lab.t().contiguous() if tn else lab, pl, ll, label_layout="TN" if tn else "NT",
                             fused_training="recompute")
        (loss * torch.tensor(head, device=dev, dtype=torch.float32)).sum().backward()
        out.append((loss.detach(), th.grad, tw.grad, tb.grad))
    for a, b_, what in zip(out[0], out[1], ("loss", "d hidden", "d weight", "d bias")):
        assert torch.equal(a, b_), what


# ---- 5. randomised agreement with the logits path -----------------------------------------------------------------------
def test_random_shapes_against_the_logits_path(dev):
    """40 random problems drawn like scripts/proj_stress.py (ragged, zero and infeasible lengths, fp32 / bf16 operands,
    with and without bias, CTA pairs and single CTAs, L up to 300): the recomputing path against ctcb_proj_loss_grad --
    bitwise losses, G within the bound and free of NaN, padded and infeasible rows exactly 0."""
    from gluon_e2e_asr_b200 import _lib
    rng = np.random.Generator(np.random.PCG64(2024))
    for c in range(40):
        B = int(rng.integers(1, 25)); T = int(rng.integers(1, 600)); V = int(rng.integers(65, 1200))
        K = 4 * int(rng.integers(1, 41)); L = int(rng.integers(0, min(T, 300) + 1))
        bf = bool(rng.integers(0, 2)); use_bias = bool(rng.integers(0, 2)); ctas = int(rng.integers(1, 3))
        if V <= L + 1:
            V = L + 2 + 63
        if bf:
            K = 8 * max(1, K // 8)
        Tb = rng.integers(0, T + 1, B); Tb[rng.integers(0, B)] = T
        Lb = rng.integers(0, L + 1, B)
        lab = rng.integers(1, V, (B, L))
        d = dict(label=lab.astype(np.float32), pred_lengths=Tb.astype(np.float32), label_lengths=Lb.astype(np.float32))
        h, w, bv = _weights(B, T, K, V, seed=c, bf16=bf, bias=use_bias)
        head = rng.uniform(0.5, 1.5, B)
        what = "case %d: B=%d T=%d K=%d V=%d L=%d bf16=%s bias=%s ctas=%d" % (c, B, T, K, V, L, bf, use_bias, ctas)
        ops = _operands(dev, h, w, bv, bf)
        labs = _dev_labels(dev, d)
        with _lib.options(proj_ctas=ctas):
            loss, G, _, _ = _recompute(dev, ops, *labs, head)
            loss_r, G_r, _ = _logits_path(dev, ops, *labs, head)
        l_c, G_c = _np(loss), _np(G)
        _against_logits_path(l_c, G_c, _np(loss_r), _np(G_r), head, what)
        st = O.param_layer(lab, Tb, Lb, T, V)[3]
        for b in range(B):
            assert (G_c[b, Tb[b]:] == 0).all(), what + ": padded rows of utterance %d" % b
            if st[b] & 1:
                assert l_c[b] == 0 and (G_c[b] == 0).all(), what + ": infeasible utterance %d" % b


# ---- 6. the emission floor ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", [12, 200])
def test_emission_floor(dev, L):
    """Frames where one non-label column lies 200 nats above every label column (beyond the 2^-100 floor of an emission):
    the recomputing forward (label columns in the shared-memory stash for L = 12, in the emission table for L = 200) and
    the logits-store forward flag UTT_WIDE_LOGITS on the same rows, give bit-identical losses, and G agrees within the
    bound -- both walk the same floored lattice.  No oracle claim: the oracle does not floor."""
    from gluon_e2e_asr_b200 import _lib
    B, T, K, V = 4, max(150, 3 * L + 50), 64, 300
    d = make_batch(B, T, V, L, seed=L + 5)
    c = V - 2                                       # the column that dominates its frames: nobody's label
    d["label"][d["label"] == c] = c - 1
    h, w, bv = _weights(B, T, K, V, seed=L + 6)
    h[:, :, K - 1] = 0.0
    w[:, K - 1] = 0.0
    w[c, K - 1] = 200.0
    hot = [(1, 37), (1, 80), (3, 5)]                # (utterance, frame), all below the utterances' frame counts
    for b, t in hot:
        assert t < d["pred_lengths"][b]
        h[b, t, K - 1] = 1.0
    head = np.linspace(0.5, 1.5, B)
    ops = _operands(dev, h, w, bv)
    labs = _dev_labels(dev, d)
    loss, G, st, _ = _recompute(dev, ops, *labs, head, status=True)
    loss_r, G_r, st_r = _logits_path(dev, ops, *labs, head, status=True)
    want = np.array([_lib.UTT_WIDE_LOGITS if b in (1, 3) else 0 for b in range(B)], np.int32)
    np.testing.assert_array_equal(_np(st), want, err_msg="recompute status")
    np.testing.assert_array_equal(_np(st_r), want, err_msg="logits path status")
    _against_logits_path(_np(loss), _np(G), _np(loss_r), _np(G_r), head, "floored batch")


# ---- 7. two graphs alive ---------------------------------------------------------------------------------------------------
def test_two_graphs_alive(dev):
    """Two recomputing forwards of the same shape, then the backwards in reverse order: each gradient has the bits of
    its batch's single run (each call keeps its own workspace until its backward)."""
    from gluon_e2e_asr_b200 import proj_ctc_loss
    B, T, K, V, L = 3, 150, 64, 300, 20
    batches = []
    for seed in (91, 92):
        d = make_batch(B, T, V, L, seed=seed)
        batches.append((_dev_labels(dev, d),) + _weights(B, T, K, V, seed=seed + 1))
    head = torch.tensor(np.linspace(0.5, 1.5, B), device=dev, dtype=torch.float32)

    def forward(i):
        labs, h, w, bv = batches[i]
        ops = tuple(t.requires_grad_(True) for t in _operands(dev, h, w, bv))
        return ops, proj_ctc_loss(*ops, *labs, fused_training="recompute")

    single = []
    for i in (0, 1):
        ops, loss = forward(i)
        (loss * head).sum().backward()
        single.append([loss.detach()] + [t.grad for t in ops])
    ops0, loss0 = forward(0)
    ops1, loss1 = forward(1)
    (loss1 * head).sum().backward()
    (loss0 * head).sum().backward()
    for i, (ops, loss) in enumerate(((ops0, loss0), (ops1, loss1))):
        for a, b_, what in zip([loss.detach()] + [t.grad for t in ops], single[i], ("loss", "d hidden", "d weight", "d bias")):
            assert torch.equal(a, b_), "batch %d: %s" % (i, what)


# ---- 8. single CTAs: the backward's shared memory ----------------------------------------------------------------------------
# proj_ctas=1: the backward's kernel holds 64 KB of G staging tiles more than the recomputing forward's, and its shared memory
# grows by 8 bytes per label-row word (Lp = Lmax rounded up to 4) and per 256-column vocabulary tile (NT): it fits the opt-in
# maximum while Lp + NT <= 2020.  The recomputing forward refuses a shape beyond that before anything runs.
NT_LIMIT_V = 256 * (2020 - 12)            # the widest vocabulary whose backward fits at Lmax = 12 (Lp = 12): 514048


def _forward_status(dev, ops, lab, pl, ll, keep):
    """ctcb_proj_forward without a logits buffer: (return code, launches)."""
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _Call, _alloc_ws, _stream_ptr
    from gluon_e2e_asr_b200.proj import _MetaLogits, _proj_struct
    B, T, V = ops[0].shape[0], ops[0].shape[1], ops[1].shape[0]
    call = _Call(_MetaLogits(torch.empty((B, T, V), device="meta"), dev), lab, pl, ll, False, True, False)
    ws = _alloc_ws(call, True)
    p = call.problem(torch.full((B,), NAN, device=dev))
    p.logits = None
    l = _lib.load()
    rc = l.ctcb_proj_forward(ctypes.byref(_proj_struct(*ops)), ctypes.byref(p), keep, ws.data_ptr(), ws.numel(), _stream_ptr(dev))
    torch.cuda.synchronize()
    return rc, _lib.last_launch_count(), l.ctcb_last_error()


def test_single_ctas_refuse_a_vocabulary_the_backward_cannot_take(dev):
    """Lmax = 12, proj_ctas=1: at V = NT_LIMIT_V the recomputing forward and backward run and agree with the logits path
    (loss also with the fp64 oracle); one column more (one more vocabulary tile) and the recomputing forward refuses with
    the backward's error and no launch, while the loss-only forward, whose kernel holds no staging tiles, still runs."""
    from gluon_e2e_asr_b200 import _lib
    B, T, K, L = 1, 40, 32, 12
    head = np.array([0.75])
    with _lib.options(proj_ctas=1):
        V = NT_LIMIT_V
        d = make_batch(B, T, V, L, seed=3)
        h, w, bv = _weights(B, T, K, V, seed=4)
        ops = _operands(dev, h, w, bv)
        labs = _dev_labels(dev, d)
        loss, G, _, _ = _recompute(dev, ops, *labs, head)
        loss_r, G_r, _ = _logits_path(dev, ops, *labs, head)
        _against_logits_path(_np(loss), _np(G), _np(loss_r), _np(G_r), head, "proj_ctas=1 V=%d" % V)
        lo = ctc_ref.ctc_ref(_logits64(h, w, bv), d["label"], d["pred_lengths"], d["label_lengths"], blank=0, layout="NTC",
                             dtype=np.float64, need_grad=False)[0]
        np.testing.assert_allclose(_np(loss), lo, rtol=RTOL, atol=ATOL)
        del G, G_r
        V = NT_LIMIT_V + 1
        w = np.concatenate([w, w[:1]])
        ops = _operands(dev, h, w, np.concatenate([bv, bv[:1]]))
        rc, launches, msg = _forward_status(dev, ops, *labs, keep=1)
        assert rc == _lib.CTCB_UNSUPPORTED and launches == 0, msg
        assert b"shared memory" in msg
        rc, launches, msg = _forward_status(dev, ops, *labs, keep=0)
        assert rc == _lib.CTCB_OK and launches > 0, msg


def test_single_ctas_take_the_longest_label_rows_the_forward_takes(dev):
    """The label-row side of the same bound: the walkers' emission ring of a gathered table ends at Lmax =
    GATHERED_LMAX_MAX, where the single-CTA backward needs 225 KB.  At that Lmax forward and backward run and agree with
    the logits path; one label more, and at Lmax = 2040, the forward refuses (CTCB_UNSUPPORTED, no launch) whether it
    keeps the history or not."""
    from gluon_e2e_asr_b200 import _lib
    K = 32
    with _lib.options(proj_ctas=1):
        L = GATHERED_LMAX_MAX
        B, T, V = 2, 2 * L + 41, L + 4
        d = make_batch(B, T, V, L, seed=7)
        h, w, bv = _weights(B, T, K, V, seed=8)
        ops = _operands(dev, h, w, bv)
        labs = _dev_labels(dev, d)
        head = np.array([0.75, 1.25])
        loss, G, _, _ = _recompute(dev, ops, *labs, head)
        loss_r, G_r, _ = _logits_path(dev, ops, *labs, head)
        _against_logits_path(_np(loss), _np(G), _np(loss_r), _np(G_r), head, "proj_ctas=1 Lmax=%d" % L)
        for L in (GATHERED_LMAX_MAX + 1, 2040):
            B, T, V = 1, 2 * L + 41, L + 60
            d = make_batch(B, T, V, L, seed=9, full_lengths=True)
            h, w, bv = _weights(B, T, K, V, seed=10)
            ops = _operands(dev, h, w, bv)
            for keep in (1, 0):
                rc, launches, msg = _forward_status(dev, ops, *_dev_labels(dev, d), keep=keep)
                assert rc == _lib.CTCB_UNSUPPORTED and launches == 0, (L, keep, msg)
                assert b"shared memory" in msg
