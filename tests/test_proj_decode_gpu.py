"""GPU tests of the greedy decode inside the fused projection (ctcb_proj_forward_decode, proj_ctc_eval).

The epilogue reduces each frame's row to its best and second best symbol from the values a logits store would write,
so the reference is ctcb_greedy_decode_typed (ops.greedy_decode) on the logits the SAME launch stores with
keep_for_backward = 1: tokens and lengths must match bit for bit.  The evaluation call (logits never stored) must give
the same tokens and exactly proj_ctc_loss's losses."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import ctc_oracle as O
from tests.synth import make_batch
from tests.test_proj_gpu import SHAPES, _problem, _tf32

pytestmark = pytest.mark.gpu

GARBAGE = 0x5EADBEEF


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _operands(dev, h, w, bv, dtype):
    th, tw = torch.tensor(h, device=dev), torch.tensor(w, device=dev)
    if dtype == "bf16":
        th, tw = th.bfloat16(), tw.bfloat16()
    return th, tw, (torch.tensor(bv, device=dev) if bv is not None else None)


def _decode_c(th, tw, tb, lab, pl, ll, unk, keep, blank_last=False, ws=None, toks=None, lens=None):
    """ctcb_proj_forward_decode through the C ABI.  keep: the logits are stored too (and returned)."""
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _Call, _alloc_ws, _stream_ptr
    from gluon_e2e_asr_b200.proj import _MetaLogits, _proj_struct
    B, T, _ = th.shape
    V, dev = tw.shape[0], th.device
    logits = torch.full((B, T, V), float("nan"), device=dev) if keep else None
    data = logits if keep else _MetaLogits(torch.empty((B, T, V), device="meta"), dev)
    call = _Call(data, lab, pl, ll, blank_last, True, False)
    ws = ws if ws is not None else _alloc_ws(call, keep)
    loss = torch.empty((B,), dtype=torch.float32, device=dev)
    toks = toks if toks is not None else torch.full((B, T), GARBAGE, dtype=torch.int32, device=dev)
    lens = lens if lens is not None else torch.full((B,), GARBAGE, dtype=torch.int32, device=dev)
    p = call.problem(loss)
    if not keep:
        p.logits = None
    pj = _proj_struct(th, tw, tb)
    _lib.check(_lib.load().ctcb_proj_forward_decode(ctypes.byref(pj), ctypes.byref(p), 1 if keep else 0,
                                                    -1 if unk is None else int(unk), toks.data_ptr(), lens.data_ptr(),
                                                    ws.data_ptr(), ws.numel(), _stream_ptr(dev)))
    return loss, toks, lens, logits


def _eq(a, b, what):
    np.testing.assert_array_equal(a.cpu().numpy(), b.cpu().numpy(), err_msg=what)


def _check_against_oracle(toks, lens, logits, pl, unk, blank):
    """tokens / lengths against the numpy oracle on the stored logits (ties: lowest index)."""
    lg = logits.cpu().numpy()
    ref = O.greedy_decode(lg, pl, blank) if unk is None else O.greedy_decode_unk(lg, pl, unk, blank)
    t, n = toks.cpu().numpy(), lens.cpu().numpy()
    for b, seq in enumerate(ref):
        assert n[b] == len(seq), (b, n[b], len(seq))
        assert list(t[b, :n[b]]) == list(seq), b
        assert (t[b, n[b]:] == 0).all(), b


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("ctas", [2, 1])
@pytest.mark.parametrize("shape", SHAPES)
def test_decode_matches_the_stored_logits_and_the_evaluation_call(dev, shape, ctas, dtype):
    """Partial frame tiles, partial vocabulary tiles, K tails; unk = none, a mid-vocabulary symbol, the blank.  The
    <unk> symbol and the blank get a bias boost so that both rules fire on many frames."""
    from gluon_e2e_asr_b200 import _lib, greedy_decode, proj_ctc_eval, proj_ctc_loss
    B, T, K, V, L = shape
    if dtype == "bf16":
        K = (K + 7) // 8 * 8                 # bf16 rows must be multiples of 16 bytes (K = 100 -> 104: still a K tail)
    d, h, w, bv = _problem(B, T, K, V, L, seed=B + 50)
    bv[V // 2] += 3.0
    bv[0] += 1.5
    th, tw, tb = _operands(dev, h, w, bv, dtype)
    lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
    with _lib.options(proj_ctas=ctas):
        with torch.no_grad():
            loss_ref = proj_ctc_loss(th, tw, tb, lab, pl, ll)
        for unk in (None, V // 2, 0):
            _, tk, lk, logits = _decode_c(th, tw, tb, lab, pl, ll, unk, keep=True)
            assert _lib.last_launch_count() == 4
            rt, rl = greedy_decode(logits, pl, blank=0, unk=unk)
            _eq(tk, rt, "tokens (stored logits), unk=%s" % unk)
            _eq(lk, rl, "lengths (stored logits), unk=%s" % unk)
            loss, te, le = proj_ctc_eval(th, tw, tb, lab, pl, ll, unk=unk)
            assert _lib.last_launch_count() == 4
            _eq(te, rt, "tokens (evaluation call), unk=%s" % unk)
            _eq(le, rl, "lengths (evaluation call), unk=%s" % unk)
            _eq(loss, loss_ref, "loss against proj_ctc_loss")
            assert not loss.requires_grad and not te.requires_grad
        # the <unk> rule is exercised: its symbol is the raw best of some valid frame
        am = logits.argmax(-1).cpu().numpy()
        assert any((am[b, :int(d["pred_lengths"][b])] == V // 2).any() for b in range(B))


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("ctas", [2, 1])
def test_exact_ties_go_to_the_lowest_index(dev, ctas, dtype):
    """Duplicate rows of W with equal bias: ties inside one 32-column chunk (40/45), across the two column halves of a
    tile (100/130), across 256-column tiles in the same half (150/390) and across tiles and halves (200/300/520).  The
    lowest index wins for the best symbol and for the <unk> rule's second best."""
    from gluon_e2e_asr_b200 import _lib
    B, T, K, V, L = 3, 300, 64, 600, 20
    d, h, w, bv = _problem(B, T, K, V, L, seed=77)
    groups = [(40, 45), (100, 130), (150, 390), (200, 300, 520)]
    rng = np.random.Generator(np.random.PCG64(78))
    for g in groups:
        row = _tf32(rng.standard_normal(K) / np.sqrt(K) * 3.0)
        boost = np.float32(rng.uniform(3.5, 4.0))
        for c in g:
            w[c] = row
            bv[c] = boost
    th, tw, tb = _operands(dev, h, w, bv, dtype)
    lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
    with _lib.options(proj_ctas=ctas):
        for unk in (None, 40, 100, 150, 200, 300, 0):
            _, tk, lk, logits = _decode_c(th, tw, tb, lab, pl, ll, unk, keep=True)
            lg = logits.cpu().numpy()
            for g in groups:                      # the ties are real in the stored logits
                for c in g[1:]:
                    np.testing.assert_array_equal(lg[..., c], lg[..., g[0]])
            am = lg.argmax(-1)
            for g in groups:                      # and every group wins some frames
                assert (am == g[0]).any(), g
            _check_against_oracle(tk, lk, logits, d["pred_lengths"], unk, 0)


@pytest.mark.parametrize("length_dtype", [torch.int32, torch.int64, torch.float32, torch.float64])
def test_hostile_lengths(dev, length_dtype):
    """Negative, > T, fractional (truncated) and zero data lengths in every length dtype; tokens beyond each length are
    zeros, lengths clamp like the parameter layer."""
    from gluon_e2e_asr_b200 import greedy_decode, proj_ctc_eval
    B, T, K, V, L = 6, 150, 64, 300, 12
    d, h, w, bv = _problem(B, T, K, V, L, seed=91)
    bv[0] += 1.5
    th, tw, tb = _operands(dev, h, w, bv, "f32")
    raw = np.array([-3.0, 170.0, 77.9, 0.0, 150.0, 64.2])
    pl = torch.tensor(raw, device=dev).to(length_dtype)
    lab, ll = torch.tensor(d["label"], device=dev), torch.tensor(d["label_lengths"], device=dev)
    for unk in (None, 7):
        _, tk, lk, logits = _decode_c(th, tw, tb, lab, pl, ll, unk, keep=True)
        rt, rl = greedy_decode(logits, pl, blank=0, unk=unk)
        _eq(tk, rt, "tokens")
        _eq(lk, rl, "lengths")
        _check_against_oracle(tk, lk, logits, pl.cpu().numpy(), unk, 0)
        _, te, le = proj_ctc_eval(th, tw, tb, lab, pl, ll, unk=unk)
        _eq(te, rt, "tokens (evaluation call)")
        _eq(le, rl, "lengths (evaluation call)")
    n = lk.cpu().numpy()
    assert n[0] == 0 and n[3] == 0 and (tk[0] == 0).all() and (tk[3] == 0).all()


@pytest.mark.parametrize("blank_label", ["first", "last"])
def test_no_lengths_and_blank_last(dev, blank_label):
    """pred_lengths=None (every frame counts) and the blank at V - 1 (dropped by the collapse)."""
    from gluon_e2e_asr_b200 import greedy_decode, proj_ctc_eval, proj_ctc_loss
    B, T, K, V, L = 4, 170, 64, 300, 18
    blank = 0 if blank_label == "first" else V - 1
    d = make_batch(B, T, V, L, seed=31, blank=blank)
    rng = np.random.Generator(np.random.PCG64(32))
    h = _tf32(rng.standard_normal((B, T, K)).astype(np.float32))
    w = _tf32((rng.standard_normal((V, K)) / np.sqrt(K)).astype(np.float32))
    bv = np.zeros(V, np.float32)
    bv[blank] = 2.0
    th, tw, tb = _operands(dev, h, w, bv, "f32")
    lab = torch.tensor(d["label"], device=dev)
    _, tk, lk, logits = _decode_c(th, tw, tb, lab, None, None, None, keep=True, blank_last=blank_label == "last")
    rt, rl = greedy_decode(logits, None, blank=blank)
    _eq(tk, rt, "tokens")
    _eq(lk, rl, "lengths")
    _check_against_oracle(tk, lk, logits, np.full(B, T), None, blank)
    assert (logits.argmax(-1) == blank).any()
    loss, te, le = proj_ctc_eval(th, tw, tb, lab, None, None, blank_label=blank_label)
    _eq(te, rt, "tokens (evaluation call)")
    _eq(le, rl, "lengths (evaluation call)")
    with torch.no_grad():
        _eq(loss, proj_ctc_loss(th, tw, tb, lab, None, None, blank_label=blank_label), "loss")


def test_both_launch_orders_give_the_same_outputs(dev):
    """The walkers beside the projection (default) or after it (proj_overlap=0): identical losses, tokens and lengths,
    four launches either way (metadata, projection, walkers, collapse)."""
    from gluon_e2e_asr_b200 import _lib, proj_ctc_eval
    B, T, K, V, L = 8, 400, 128, 1000, 40
    d, h, w, bv = _problem(B, T, K, V, L, seed=5)
    th, tw, tb = _operands(dev, h, w, bv, "f32")
    lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
    outs = []
    for overlap in (-1, 0):
        with _lib.options(proj_overlap=overlap):
            outs.append(proj_ctc_eval(th, tw, tb, lab, pl, ll, unk=3))
            assert _lib.last_launch_count() == 4
    for a, b, what in zip(outs[0], outs[1], ("loss", "tokens", "lengths")):
        _eq(a, b, what)


@pytest.mark.parametrize("overlap", [-1, 0])
def test_back_to_back_calls_on_one_workspace(dev, overlap):
    """Two evaluation calls with different inputs on one workspace and one pair of output buffers, enqueued without a
    synchronisation in between, outputs pre-filled with garbage: each matches its own reference (tile flags left set by
    the first call must not let the second call's collapse run ahead of its projection)."""
    from gluon_e2e_asr_b200 import _lib, greedy_decode
    B, T, K, V, L = 6, 500, 256, 2000, 60
    probs = []
    for seed in (1, 2):
        d, h, w, bv = _problem(B, T, K, V, L, seed=seed)
        th, tw, tb = _operands(dev, h, w, bv, "f32")
        lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
        _, _, _, logits = _decode_c(th, tw, tb, lab, pl, ll, None, keep=True)
        probs.append((th, tw, tb, lab, pl, ll, greedy_decode(logits, pl, blank=0)))
    ws = torch.empty((_lib.workspace_bytes(T, B, V, L, False),), dtype=torch.uint8, device=dev)
    toks = torch.full((B, T), GARBAGE, dtype=torch.int32, device=dev)
    lens = torch.full((B,), GARBAGE, dtype=torch.int32, device=dev)
    with _lib.options(proj_overlap=overlap):
        got = []
        for th, tw, tb, lab, pl, ll, _ in probs:
            _decode_c(th, tw, tb, lab, pl, ll, None, keep=False, ws=ws, toks=toks, lens=lens)
            got.append((toks.clone(), lens.clone()))
            toks.fill_(GARBAGE)
            lens.fill_(GARBAGE)
    for (t, n), pr in zip(got, probs):
        rt, rl = pr[-1]
        _eq(t, rt, "tokens")
        _eq(n, rl, "lengths")


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_wer_totals_match_the_library_gemm_path(dev, dtype):
    """edit_distance over the fused hypotheses against edit_distance over ops.greedy_decode of library-GEMM logits.  The
    operands are small multiples of 1/2 and the bias of 1/4: every product and sum is exact in fp32 (and bf16 operands),
    so both logits tensors are identical whatever the accumulation order, and so are the hypotheses."""
    from gluon_e2e_asr_b200 import edit_distance, greedy_decode, proj_ctc_eval
    B, T, K, V, L = 8, 500, 64, 2000, 60
    d = make_batch(B, T, V, L, seed=3)
    rng = np.random.Generator(np.random.PCG64(4))
    h = (rng.integers(-2, 3, (B, T, K)) * 0.5).astype(np.float32)
    w = rng.integers(-1, 2, (V, K)).astype(np.float32)
    bv = (rng.integers(-4, 5, V) * 0.25).astype(np.float32)
    bv[0] = 4.0                                        # blanks on many frames, as in a trained model
    th, tw, tb = _operands(dev, h, w, bv, dtype)
    lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
    _, toks, lens = proj_ctc_eval(th, tw, tb, lab, pl, ll)
    logits = torch.nn.functional.linear(th.float(), tw.float(), tb)
    rt, rl = greedy_decode(logits, pl, blank=0)
    ref = lab.to(torch.int32).contiguous()
    rlen = ll.to(torch.int32).contiguous()
    tot_f = torch.zeros(2, dtype=torch.int64, device=dev)
    tot_r = torch.zeros(2, dtype=torch.int64, device=dev)
    dist_f = edit_distance(ref, rlen, toks, lens, tot_f)
    dist_r = edit_distance(ref, rlen, rt, rl, tot_r)
    _eq(dist_f, dist_r, "per-utterance distances")
    _eq(tot_f, tot_r, "WER totals")
    _eq(toks, rt, "tokens")
    assert int(tot_f[1]) == int(d["label_lengths"].sum()) and int(rl.sum()) > 0
