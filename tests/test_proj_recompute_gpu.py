"""GPU parity of the recomputing training path of the fused projection (proj_ctc_loss(..., fused_training="recompute"):
ctcb_proj_forward with keep_for_backward and no logits buffer, then ctcb_proj_backward) against  oracle ∘ fp64 matmul,
against fused_training=True, and against ctcb_proj_loss_grad's d loss / d logits on the same operands.

Helpers are copies of test_proj_gpu.py's (tf32-representable inputs: the products are exact, so the path must meet the
logits path's bar, rtol 1e-4 / atol 1e-5 against the fp64 oracle of the fp64 product)."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import ctc_ref
from tests.synth import make_batch

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-4, 1e-5
TF32_REL = 4e-3                           # d hidden / d weight: tf32 library GEMMs of the (fp32) logit gradient, norm-wise
BF16_REL = 1e-2                           # ... returned in bfloat16 for bfloat16 operands
# G against ctcb_proj_loss_grad's: the softmax part is the same MMA sequence and the same fp32 arithmetic (bit-identical);
# the occupancies come from the same 20-bit-mantissa high words of the walkers' history, normalised per frame by their sum
# there and by P(l|x) of frame 0 here -- two normalisers that agree to the history's 2^-20.  Hence |dG| <= 4e-6 |head|.
G_VS_LOGITS_PATH = 4e-6


def _close_tf32(actual, desired, what, rel=TF32_REL):
    err, scale = np.abs(actual - desired).max(), np.abs(desired).max()
    assert err <= rel * scale, "%s: max error %.3e against scale %.3e" % (what, err, scale)


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _tf32(x):
    return (np.ascontiguousarray(x, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def _problem(B, T, K, V, L, seed, exact=True, bias=True, full_lengths=False):
    d = make_batch(B, T, V, L, seed=seed, full_lengths=full_lengths)
    rng = np.random.Generator(np.random.PCG64(seed + 1000))
    h = rng.standard_normal((B, T, K)).astype(np.float32)
    w = (rng.standard_normal((V, K)) / np.sqrt(K)).astype(np.float32)
    bv = (rng.standard_normal((V,)) * 0.5).astype(np.float32) if bias else None
    if exact:
        h, w = _tf32(h), _tf32(w)
    return d, h, w, bv


def _oracle(d, h, w, bv, head, blank=0, check_feasible=True):
    logits = h.astype(np.float64) @ w.astype(np.float64).T
    if bv is not None:
        logits = logits + bv.astype(np.float64)
    lo, G, feas = ctc_ref.ctc_ref(logits, d["label"], d["pred_lengths"], d["label_lengths"], blank=blank, head_grad=head,
                                  layout="NTC", dtype=np.float64)
    if check_feasible:
        assert feas.all()
    for b in range(G.shape[0]):                      # padded frames: exact zeros
        G[b, int(d["pred_lengths"][b]):] = 0.0
        if not feas[b]:
            G[b] = 0.0
    G2 = G.reshape(-1, G.shape[2])
    dh = (G2 @ w.astype(np.float64)).reshape(h.shape)
    dw = G2.T @ h.astype(np.float64).reshape(-1, h.shape[2])
    db = G2.sum(0)
    return lo, G, dh, dw, db


def _operands(dev, h, w, bv, bf16):
    th, tw = torch.tensor(h, device=dev), torch.tensor(w, device=dev)
    if bf16:
        th, tw = th.bfloat16(), tw.bfloat16()
    tb = torch.tensor(bv, device=dev) if bv is not None else None
    return th, tw, tb


def _run(dev, d, h, w, bv, head, fused_training="recompute", bf16=False):
    """autograd: loss, d hidden, d weight, d bias (fp32 numpy)."""
    from gluon_e2e_asr_b200 import proj_ctc_loss
    th, tw, tb = _operands(dev, h, w, bv, bf16)
    for t in (th, tw, tb):
        if t is not None:
            t.requires_grad_(True)
    lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
    loss = proj_ctc_loss(th, tw, tb, lab, pl, ll, fused_training=fused_training)
    (loss * torch.tensor(head, device=dev, dtype=torch.float32)).sum().backward()
    return (loss.detach().cpu().numpy(), th.grad.float().cpu().numpy(), tw.grad.float().cpu().numpy(),
            tb.grad.cpu().numpy() if tb is not None else None)


def _abi(dev, d, h, w, bv, head, bf16=False, reference=True, lengths=True):
    """Through the C ABI: (loss, G) of ctcb_proj_forward(keep, no logits) + ctcb_proj_backward into a NaN-poisoned G, and
    (loss, G) of ctcb_proj_loss_grad on the same operands (reference=True)."""
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _Call, _alloc_ws, _stream_ptr
    from gluon_e2e_asr_b200.proj import _MetaLogits, _proj_struct
    B, T, _ = h.shape
    V = w.shape[0]
    th, tw, tb = _operands(dev, h, w, bv, bf16)
    lab = torch.tensor(d["label"], device=dev)
    pl = torch.tensor(d["pred_lengths"], device=dev) if lengths else None
    ll = torch.tensor(d["label_lengths"], device=dev) if lengths else None
    hd = torch.tensor(head, device=dev, dtype=torch.float32)
    l = _lib.load()
    pj = _proj_struct(th, tw, tb)
    call = _Call(_MetaLogits(torch.empty((B, T, V), device="meta"), dev), lab, pl, ll, False, True, False)
    ws = _alloc_ws(call, True)
    loss = torch.empty((B,), device=dev)
    p = call.problem(loss)
    p.logits = None
    _lib.check(l.ctcb_proj_forward(ctypes.byref(pj), ctypes.byref(p), 1, ws.data_ptr(), ws.numel(), _stream_ptr(dev)))
    assert _lib.last_launch_count() == 4          # k_proj_emit, metadata, k_walk, k_proj_occ
    G = torch.full((B, T, V), float("nan"), device=dev)
    scratch = torch.empty((B,), device=dev)
    p2 = call.problem(scratch, grad=G, head=hd)
    p2.logits = None
    _lib.check(l.ctcb_proj_backward(ctypes.byref(pj), ctypes.byref(p2), ws.data_ptr(), ws.numel(), _stream_ptr(dev)))
    assert _lib.last_launch_count() == 1
    out = [loss.cpu().numpy(), G.cpu().numpy()]
    if reference:
        logits = torch.empty((B, T, V), device=dev)
        Gr = torch.empty_like(logits)
        loss_r = torch.empty((B,), device=dev)
        call_r = _Call(logits, lab, pl, ll, False, True, False)
        ws_r = _alloc_ws(call_r, True)
        pr = call_r.problem(loss_r, Gr, hd)
        _lib.check(l.ctcb_proj_loss_grad(ctypes.byref(pj), ctypes.byref(pr), ws_r.data_ptr(), ws_r.numel(), _stream_ptr(dev)))
        out += [loss_r.cpu().numpy(), Gr.cpu().numpy()]
    torch.cuda.synchronize()
    return out


SHAPES = [
    # B, T, K, V, L        -- test_proj_gpu.py's shapes
    (3, 150, 64, 300, 20),       # two frame tiles (second partial), two vocabulary tiles (second partial), two K blocks
    (2, 128, 32, 256, 10),       # exactly one tile each way, one K block
    (4, 300, 100, 520, 33),      # K not a multiple of 32 (zero-filled tail), three vocabulary tiles
    (5, 97, 256, 1000, 40),      # deep K loop: the ring wraps several times
]


@pytest.mark.parametrize("bf16", [False, True], ids=["fp32", "bf16"])
@pytest.mark.parametrize("ctas", [2, 1])
@pytest.mark.parametrize("shape", SHAPES)
def test_recompute_matches_oracle_and_the_logits_paths(dev, shape, ctas, bf16):
    """Loss and G (C ABI) against the fp64 oracle of the fp64 product of the operands as the kernel sees them; losses
    bit-identical to fused_training=True; G against ctcb_proj_loss_grad's; d hidden / d weight / d bias at the tf32
    contractions' bar.  Non-uniform head."""
    from gluon_e2e_asr_b200 import _lib
    B, T, K, V, L = shape
    if bf16:
        K = (K + 7) // 8 * 8                       # bfloat16 rows: K a multiple of 8 (16 bytes); 100 -> 104
    d, h, w, bv = _problem(B, T, K, V, L, seed=B + 17, exact=not bf16)
    if bf16:                                       # the oracle of the bfloat16 values the kernel multiplies
        h = torch.tensor(h).bfloat16().float().numpy()
        w = torch.tensor(w).bfloat16().float().numpy()
    head = np.linspace(0.5, 1.5, B)
    lo, G, dh, dw, db = _oracle(d, h, w, bv, head)
    with _lib.options(proj_ctas=ctas):
        loss_c, G_c, loss_r, G_r = _abi(dev, d, h, w, bv, head, bf16=bf16)
        loss, gh, gw, gb = _run(dev, d, h, w, bv, head, bf16=bf16)
        loss_t, _, _, _ = _run(dev, d, h, w, bv, head, fused_training=True, bf16=bf16)
    np.testing.assert_allclose(loss, lo, rtol=RTOL, atol=ATOL, err_msg="loss")
    np.testing.assert_array_equal(loss, loss_t, err_msg="losses of fused_training=True")
    np.testing.assert_array_equal(loss_c, loss)
    np.testing.assert_array_equal(loss_r, loss)
    np.testing.assert_allclose(G_c, G, rtol=RTOL, atol=ATOL, err_msg="d logits")
    np.testing.assert_allclose(G_c, G_r, rtol=0, atol=G_VS_LOGITS_PATH * head.max(), err_msg="d logits vs logits path")
    rel = BF16_REL if bf16 else TF32_REL
    _close_tf32(gh, dh, "d hidden", rel)
    _close_tf32(gw, dw, "d weight", rel)
    np.testing.assert_allclose(gb, db, rtol=2e-3, atol=2e-4, err_msg="d bias")


@pytest.mark.parametrize("blank_label", ["first", "last"])
def test_blank_last_and_inferred_lengths(dev, blank_label):
    """No length vectors: T frames per utterance, labels end at the first padding value; blank 'last' lies in the last
    vocabulary tile's partial half."""
    from gluon_e2e_asr_b200 import proj_ctc_loss
    from oracle import ctc_oracle as O
    B, T, K, V, L = 4, 170, 64, 300, 18
    blank = 0 if blank_label == "first" else V - 1
    d = make_batch(B, T, V, L, seed=31, blank=blank)
    rng = np.random.Generator(np.random.PCG64(32))
    h = _tf32(rng.standard_normal((B, T, K)).astype(np.float32))
    w = _tf32((rng.standard_normal((V, K)) / np.sqrt(K)).astype(np.float32))
    logits = h.astype(np.float64) @ w.astype(np.float64).T
    head = np.array([1.0, 0.5, 2.0, 0.25])
    lo, G, ok = O.CtcLossOracle("NTC", "NT", blank_label)(logits, d["label"], None, None, head_grad=head)
    assert ok.all()
    th, tw = torch.tensor(h, device=dev, requires_grad=True), torch.tensor(w, device=dev, requires_grad=True)
    loss = proj_ctc_loss(th, tw, None, torch.tensor(d["label"], device=dev), None, None, blank_label=blank_label,
                         fused_training="recompute")
    (loss * torch.tensor(head, device=dev, dtype=torch.float32)).sum().backward()
    np.testing.assert_allclose(loss.detach().cpu().numpy(), lo, rtol=RTOL, atol=ATOL)
    G2 = np.asarray(G, np.float64).reshape(-1, V)
    _close_tf32(th.grad.cpu().numpy(), (G2 @ w.astype(np.float64)).reshape(h.shape), "d hidden")
    _close_tf32(tw.grad.cpu().numpy(), G2.T @ h.astype(np.float64).reshape(-1, K), "d weight")


@pytest.mark.parametrize("case", ["long_labels", "v_not_multiple_of_4", "no_bias"])
def test_layout_corners(dev, case):
    """Label rows too long for the shared-memory stash (321 columns: parked in the emission table, which the occupancy
    table then replaces); V not a multiple of 4 (no 16-byte bias loads, G rows without a tensor map: coalesced row
    stores); no bias."""
    shape, kw = {"long_labels": ((2, 700, 32, 600, 320), dict(full_lengths=True)),
                 "v_not_multiple_of_4": ((3, 200, 64, 301, 20), {}),
                 "no_bias": ((3, 180, 64, 400, 25), dict(bias=False))}[case]
    B, T, K, V, L = shape
    d, h, w, bv = _problem(B, T, K, V, L, seed=43, **kw)
    head = np.linspace(1.5, 0.5, B)
    lo, G, dh, dw, db = _oracle(d, h, w, bv, head)
    loss_c, G_c, _, G_r = _abi(dev, d, h, w, bv, head)
    np.testing.assert_allclose(loss_c, lo, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(G_c, G, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(G_c, G_r, rtol=0, atol=G_VS_LOGITS_PATH * head.max())
    loss, gh, gw, gb = _run(dev, d, h, w, bv, head)
    np.testing.assert_array_equal(loss, loss_c)
    _close_tf32(gh, dh, "d hidden")
    _close_tf32(gw, dw, "d weight")
    if bv is None:
        assert gb is None
    else:
        np.testing.assert_allclose(gb, db, rtol=2e-3, atol=2e-4)


def test_padded_tiles_infeasible_and_empty_utterances(dev):
    """pred_lengths far below T (whole 128-frame tiles, and CTA pairs, of padding): those G rows are exactly 0 in a
    NaN-poisoned buffer; an empty utterance (T_b = 0) and an infeasible one (L_b > T_b) have loss 0 and G = 0."""
    B, T, K, V, L = 5, 700, 64, 300, 12
    d, h, w, bv = _problem(B, T, K, V, L, seed=51)
    d["pred_lengths"] = np.array([40, 700, 0, 5, 130], np.float32)
    d["label_lengths"] = np.array([12, 12, 3, 9, 1], np.float32)        # utterance 3: 9 labels in 5 frames
    head = np.linspace(0.5, 1.5, B)
    lo, G, dh, dw, db = _oracle(d, h, w, bv, head, check_feasible=False)
    loss_c, G_c, loss_r, G_r = _abi(dev, d, h, w, bv, head)
    assert loss_c[2] == 0.0 and loss_c[3] == 0.0
    assert (G_c[2] == 0).all() and (G_c[3] == 0).all()
    for b, tb in enumerate(d["pred_lengths"].astype(int)):
        assert (G_c[b, tb:] == 0).all(), "padded rows of utterance %d" % b
    live = [0, 1, 4]
    np.testing.assert_allclose(loss_c[live], lo[live], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(G_c, G, rtol=RTOL, atol=ATOL)
    np.testing.assert_array_equal(loss_c, loss_r)
    np.testing.assert_allclose(G_c, G_r, rtol=0, atol=G_VS_LOGITS_PATH * head.max())


def test_second_backward_raises(dev):
    from gluon_e2e_asr_b200 import proj_ctc_loss
    B, T, K, V, L = 2, 128, 32, 256, 10
    d, h, w, bv = _problem(B, T, K, V, L, seed=61)
    th = torch.tensor(h, device=dev, requires_grad=True)
    tw = torch.tensor(w, device=dev)
    lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
    loss = proj_ctc_loss(th, tw, None, lab, pl, ll, fused_training="recompute")
    loss.sum().backward(retain_graph=True)
    with pytest.raises(RuntimeError):
        loss.sum().backward()


def test_backward_on_a_workspace_no_forward_filled_gives_nan(dev):
    """A zeroed workspace, and one filled by a loss-only forward (another layout stamp): NaN rows, no wait."""
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _Call, _alloc_ws, _stream_ptr
    from gluon_e2e_asr_b200.proj import _MetaLogits, _proj_struct
    B, T, K, V, L = 3, 150, 64, 300, 20
    d, h, w, bv = _problem(B, T, K, V, L, seed=71)
    th, tw, tb = _operands(dev, h, w, bv, False)
    lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
    l = _lib.load()
    pj = _proj_struct(th, tw, tb)
    call = _Call(_MetaLogits(torch.empty((B, T, V), device="meta"), dev), lab, pl, ll, False, True, False)
    ws = _alloc_ws(call, True)
    for fill_with_loss_only_forward in (False, True):
        ws.zero_()
        loss = torch.empty((B,), device=dev)
        if fill_with_loss_only_forward:
            p = call.problem(loss)
            p.logits = None
            _lib.check(l.ctcb_proj_forward(ctypes.byref(pj), ctypes.byref(p), 0, ws.data_ptr(), ws.numel(), _stream_ptr(dev)))
        G = torch.zeros((B, T, V), device=dev)
        p2 = call.problem(loss, grad=G)
        p2.logits = None
        _lib.check(l.ctcb_proj_backward(ctypes.byref(pj), ctypes.byref(p2), ws.data_ptr(), ws.numel(), _stream_ptr(dev)))
        torch.cuda.synchronize()
        assert torch.isnan(G).all()


def test_cfg3_shape(dev):
    """BASELINE configs[2] with H = 512 at its batch of 64: loss against the oracle, losses bit-identical to
    fused_training=True, G against ctcb_proj_loss_grad's, parameter gradients against the fused_training=True path."""
    B, T, K, V, L = 64, 500, 512, 2000, 150
    d, h, w, bv = _problem(B, T, K, V, L, seed=11)
    head = np.full(B, 1.0 / B)
    logits = h.astype(np.float64) @ w.astype(np.float64).T + bv.astype(np.float64)
    lo, _, feas = ctc_ref.ctc_ref(logits, d["label"], d["pred_lengths"], d["label_lengths"], blank=0, head_grad=head,
                                  layout="NTC", dtype=np.float64)
    del logits
    assert feas.all()
    loss_c, G_c, loss_r, G_r = _abi(dev, d, h, w, bv, head)
    np.testing.assert_allclose(loss_c, lo, rtol=RTOL, atol=ATOL)
    np.testing.assert_array_equal(loss_c, loss_r)
    np.testing.assert_allclose(G_c, G_r, rtol=0, atol=G_VS_LOGITS_PATH * head.max())
    del G_c, G_r
    loss, gh, gw, gb = _run(dev, d, h, w, bv, head)
    loss_t, gh_t, gw_t, gb_t = _run(dev, d, h, w, bv, head, fused_training=True)
    np.testing.assert_array_equal(loss, loss_t)
    _close_tf32(gh, gh_t, "d hidden")
    _close_tf32(gw, gw_t, "d weight")
    np.testing.assert_allclose(gb, gb_t, rtol=2e-3, atol=2e-4)
