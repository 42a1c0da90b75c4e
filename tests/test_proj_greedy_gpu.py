"""GPU tests of the label-free greedy decode from the encoder output (ctcb_proj_greedy_decode, proj_greedy_decode,
ProjCtcLoss.decode).

The decode-only epilogue forms each frame's word exactly as the loss + decode epilogue does, from the same accumulator
tiles in the same K order, so the reference is proj_ctc_eval (whatever labels it gets): tokens and lengths must match bit
for bit, and through it ctcb_greedy_decode_unk on the logits the projection stores.  Where proj_ctc_eval refuses
(V <= 64), exactly representable operands make every logits tensor identical, and the reference is greedy_decode of
torch.nn.functional.linear."""
import ctypes

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from tests.synth import make_batch
from tests.test_proj_decode_gpu import GARBAGE, _check_against_oracle, _decode_c, _eq, _operands
from tests.test_proj_gpu import SHAPES, _problem, _tf32

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _greedy_c(th, tw, tb, pl, blank, unk, toks, lens):
    """ctcb_proj_greedy_decode through the C ABI into the caller's output buffers."""
    from gluon_e2e_asr_b200 import _lib
    from gluon_e2e_asr_b200.ops import _DT, _stream_ptr
    from gluon_e2e_asr_b200.proj import _proj_struct
    B, T, _ = th.shape
    pj = _proj_struct(th, tw, tb)
    _lib.check(_lib.load().ctcb_proj_greedy_decode(ctypes.byref(pj), T, B, tw.shape[0],
                                                   pl.data_ptr() if pl is not None else None,
                                                   _DT[pl.dtype] if pl is not None else 0, blank,
                                                   -1 if unk is None else int(unk), toks.data_ptr(), lens.data_ptr(),
                                                   _stream_ptr(th.device)))


def _exact(B, T, K, V, seed, dtype, dev):
    """Operands whose every product and partial sum is exact in fp32 (and bf16 operands): halves times {-1, 0, 1},
    bias in quarters -- the logits are the same whatever GEMM forms them (ties included)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    h = (rng.integers(-2, 3, (B, T, K)) * 0.5).astype(np.float32)
    w = rng.integers(-1, 2, (V, K)).astype(np.float32)
    bv = (rng.integers(-4, 5, V) * 0.25).astype(np.float32)
    bv[0] = 2.0                                        # blanks on many frames
    return _operands(dev, h, w, bv, dtype)


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("ctas", [2, 1])
@pytest.mark.parametrize("shape", SHAPES)
def test_decode_matches_the_evaluation_call(dev, shape, ctas, dtype):
    """Every projection test shape (partial frame and vocabulary tiles, K tails, deep K loops); unk = none, a
    mid-vocabulary symbol (boosted so that the rule fires), the blank.  Two launches; equal to proj_ctc_eval and to
    greedy_decode on the logits ctcb_proj_forward_decode stores."""
    from gluon_e2e_asr_b200 import _lib, greedy_decode, proj_ctc_eval, proj_greedy_decode
    B, T, K, V, L = shape
    if dtype == "bf16":
        K = (K + 7) // 8 * 8
    d, h, w, bv = _problem(B, T, K, V, L, seed=B + 60)
    bv[V // 2] += 3.0
    bv[0] += 1.5
    th, tw, tb = _operands(dev, h, w, bv, dtype)
    lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
    with _lib.options(proj_ctas=ctas):
        for unk in (None, V // 2, 0):
            tk, lk = proj_greedy_decode(th, tw, tb, pl, unk=unk)
            assert _lib.last_launch_count() == 2
            assert tk.dtype == torch.int32 and lk.dtype == torch.int32 and not tk.requires_grad
            _, te, le = proj_ctc_eval(th, tw, tb, lab, pl, ll, unk=unk)
            _eq(tk, te, "tokens against proj_ctc_eval, unk=%s" % unk)
            _eq(lk, le, "lengths against proj_ctc_eval, unk=%s" % unk)
            _, _, _, logits = _decode_c(th, tw, tb, lab, pl, ll, unk, keep=True)
            rt, rl = greedy_decode(logits, pl, blank=0, unk=unk)
            _eq(tk, rt, "tokens against the stored logits, unk=%s" % unk)
            _eq(lk, rl, "lengths against the stored logits, unk=%s" % unk)
        am = logits.argmax(-1).cpu().numpy()
        assert any((am[b, :int(d["pred_lengths"][b])] == V // 2).any() for b in range(B))


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("ctas", [2, 1])
def test_exact_ties_go_to_the_lowest_index(dev, ctas, dtype):
    """Duplicate rows of W with equal bias: ties inside one 32-column chunk (40/45), across the two column halves of a
    tile (100/130), across 256-column tiles (150/390) and across tiles and halves (200/300/520)."""
    from gluon_e2e_asr_b200 import _lib, proj_ctc_eval, proj_greedy_decode
    B, T, K, V, L = 3, 300, 64, 600, 20
    d, h, w, bv = _problem(B, T, K, V, L, seed=79)
    groups = [(40, 45), (100, 130), (150, 390), (200, 300, 520)]
    rng = np.random.Generator(np.random.PCG64(80))
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
            tk, lk = proj_greedy_decode(th, tw, tb, pl, unk=unk)
            _, te, le = proj_ctc_eval(th, tw, tb, lab, pl, ll, unk=unk)
            _eq(tk, te, "tokens, unk=%s" % unk)
            _eq(lk, le, "lengths, unk=%s" % unk)
            _, _, _, logits = _decode_c(th, tw, tb, lab, pl, ll, unk, keep=True)
            am = logits.argmax(-1).cpu().numpy()
            for g in groups:                      # every group wins some frames
                assert (am == g[0]).any(), g
            _check_against_oracle(tk, lk, logits, d["pred_lengths"], unk, 0)


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("ctas", [2, 1])
@pytest.mark.parametrize("V", [46, 64, 301])
def test_small_and_odd_vocabularies_match_torch_logits(dev, V, ctas, dtype):
    """V = 46 (the character vocabulary of the small shapes) and V = 64, where the fused loss refuses, and V = 301; 46 and
    301 are not multiples of 4 (the scalar bias path).  Exactly representable operands: bit-exact against greedy_decode
    of torch.nn.functional.linear, whose lowest-index tie rule the kernel shares."""
    from gluon_e2e_asr_b200 import _lib, greedy_decode, proj_greedy_decode
    B, T, K = 5, 300, 64
    th, tw, tb = _exact(B, T, K, V, seed=V + ctas, dtype=dtype, dev=dev)
    pl = torch.tensor(make_batch(B, T, V, 8, seed=V)["pred_lengths"], device=dev)
    logits = torch.nn.functional.linear(th.float(), tw.float(), tb)
    with _lib.options(proj_ctas=ctas):
        for unk in (None, V // 3, 0):
            tk, lk = proj_greedy_decode(th, tw, tb, pl, unk=unk)
            rt, rl = greedy_decode(logits, pl, blank=0, unk=unk)
            _eq(tk, rt, "tokens, unk=%s" % unk)
            _eq(lk, rl, "lengths, unk=%s" % unk)
            _check_against_oracle(tk, lk, logits, pl.cpu().numpy(), unk, 0)
    assert int(lk.sum()) > 0


@pytest.mark.parametrize("length_dtype", [torch.int32, torch.int64, torch.float32, torch.float64])
def test_hostile_lengths(dev, length_dtype):
    """Negative, > T, fractional (truncated) and zero lengths in every length dtype: lengths clamp like the parameter
    layer, tokens beyond each hypothesis are zeros; equal to proj_ctc_eval with the same lengths."""
    from gluon_e2e_asr_b200 import greedy_decode, proj_ctc_eval, proj_greedy_decode
    B, T, K, V, L = 6, 150, 64, 300, 12
    d, h, w, bv = _problem(B, T, K, V, L, seed=93)
    bv[0] += 1.5
    th, tw, tb = _operands(dev, h, w, bv, "f32")
    pl = torch.tensor(np.array([-3.0, 170.0, 77.9, 0.0, 150.0, 64.2]), device=dev).to(length_dtype)
    lab, ll = torch.tensor(d["label"], device=dev), torch.tensor(d["label_lengths"], device=dev)
    for unk in (None, 7):
        tk, lk = proj_greedy_decode(th, tw, tb, pl, unk=unk)
        _, te, le = proj_ctc_eval(th, tw, tb, lab, pl, ll, unk=unk)
        _eq(tk, te, "tokens")
        _eq(lk, le, "lengths")
        _, _, _, logits = _decode_c(th, tw, tb, lab, pl, ll, unk, keep=True)
        rt, rl = greedy_decode(logits, pl, blank=0, unk=unk)
        _eq(tk, rt, "tokens against the stored logits")
        _eq(lk, rl, "lengths against the stored logits")
    n = lk.cpu().numpy()
    assert n[0] == 0 and n[3] == 0 and (tk[0] == 0).all() and (tk[3] == 0).all()


@pytest.mark.parametrize("blank_label", ["first", "last"])
def test_no_lengths_and_the_block_blank(dev, blank_label):
    """pred_lengths=None (every frame counts), through ProjCtcLoss.decode, whose blank is the block's (V - 1 for
    blank_label="last"): equal to ProjCtcLoss.evaluate."""
    from gluon_e2e_asr_b200 import ProjCtcLoss, proj_greedy_decode
    B, T, K, V, L = 4, 170, 64, 300, 18
    blank = 0 if blank_label == "first" else V - 1
    d = make_batch(B, T, V, L, seed=33, blank=blank)
    rng = np.random.Generator(np.random.PCG64(34))
    block = ProjCtcLoss(K, V, blank_label=blank_label).to(dev)
    with torch.no_grad():
        block.weight.copy_(torch.tensor(_tf32(rng.standard_normal((V, K)) / np.sqrt(K)), device=dev))
        block.bias.zero_()
        block.bias[blank] = 2.0
    th = torch.tensor(_tf32(rng.standard_normal((B, T, K)).astype(np.float32)), device=dev)
    lab = torch.tensor(d["label"], device=dev)
    tk, lk = block.decode(th)
    _, te, le = block.evaluate(th, lab)
    _eq(tk, te, "tokens")
    _eq(lk, le, "lengths")
    t2, l2 = proj_greedy_decode(th, block.weight, block.bias, blank=blank)
    _eq(tk, t2, "tokens (function)")
    _eq(lk, l2, "lengths (function)")
    assert not tk.requires_grad and int(lk.sum()) > 0
    if blank:
        assert (tk != blank).all()                     # dropped by the collapse


def test_tnc_strided_hidden_and_no_bias(dev):
    """hidden as a (B, T, K) view of a (T, B, K) buffer (the operator's TNC layout), and bias=None: equal to the
    contiguous call and to proj_ctc_eval."""
    from gluon_e2e_asr_b200 import proj_ctc_eval, proj_greedy_decode
    B, T, K, V, L = 4, 260, 96, 700, 25
    d, h, w, _ = _problem(B, T, K, V, L, seed=17, bias=False)
    th, tw, _ = _operands(dev, h, w, None, "f32")
    tnc = th.transpose(0, 1).contiguous().transpose(0, 1)
    assert tnc.stride() == (K, B * K, 1)
    lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
    for unk in (None, 5):
        tk, lk = proj_greedy_decode(tnc, tw, None, pl, unk=unk)
        tc, lc = proj_greedy_decode(th, tw, None, pl, unk=unk)
        _, te, le = proj_ctc_eval(th, tw, None, lab, pl, ll, unk=unk)
        _eq(tk, tc, "tokens (strided against contiguous)")
        _eq(lk, lc, "lengths (strided against contiguous)")
        _eq(tk, te, "tokens against proj_ctc_eval")
        _eq(lk, le, "lengths against proj_ctc_eval")


def test_back_to_back_calls_into_garbage_filled_outputs(dev):
    """Two decodes with different inputs into one pair of output buffers pre-filled with garbage, enqueued without a
    synchronisation in between: each matches its own reference (prefix, zeros after it, length)."""
    from gluon_e2e_asr_b200 import proj_ctc_eval
    B, T, K, V, L = 6, 500, 256, 2000, 60
    probs = []
    for seed in (1, 2):
        d, h, w, bv = _problem(B, T, K, V, L, seed=seed)
        th, tw, tb = _operands(dev, h, w, bv, "f32")
        lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
        probs.append((th, tw, tb, pl, proj_ctc_eval(th, tw, tb, lab, pl, ll, unk=9)[1:]))
    toks = torch.full((B, T), GARBAGE, dtype=torch.int32, device=dev)
    lens = torch.full((B,), GARBAGE, dtype=torch.int32, device=dev)
    got = []
    for th, tw, tb, pl, _ in probs:
        _greedy_c(th, tw, tb, pl, 0, 9, toks, lens)
        got.append((toks.clone(), lens.clone()))
        toks.fill_(GARBAGE)
        lens.fill_(GARBAGE)
    for (t, n), pr in zip(got, probs):
        rt, rl = pr[-1]
        _eq(t, rt, "tokens")
        _eq(n, rl, "lengths")


def test_a_decode_right_after_an_evaluation_on_the_same_stream(dev):
    """proj_ctc_eval leaves the tile flags of its workspace set and its walkers may still run when the next call is
    enqueued: a decode enqueued right behind it (and an evaluation right behind the decode) gives the outputs it gives
    alone."""
    from gluon_e2e_asr_b200 import proj_ctc_eval, proj_greedy_decode
    B, T, K, V, L = 8, 400, 128, 1000, 40
    d, h, w, bv = _problem(B, T, K, V, L, seed=6)
    th, tw, tb = _operands(dev, h, w, bv, "f32")
    lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
    alone = proj_greedy_decode(th, tw, tb, pl, unk=3)
    eval_alone = proj_ctc_eval(th, tw, tb, lab, pl, ll, unk=3)
    torch.cuda.synchronize()
    e1 = proj_ctc_eval(th, tw, tb, lab, pl, ll, unk=3)
    g1 = proj_greedy_decode(th, tw, tb, pl, unk=3)
    e2 = proj_ctc_eval(th, tw, tb, lab, pl, ll, unk=3)
    for a, b, what in zip(alone, g1, ("tokens", "lengths")):
        _eq(a, b, what)
    for run in (e1, e2):
        for a, b, what in zip(eval_alone, run, ("loss", "tokens", "lengths")):
            _eq(a, b, what)


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("V", [46, 2000])
def test_wer_totals_match_the_library_gemm_path(dev, V, dtype):
    """edit_distance over the decoded hypotheses against edit_distance over ops.greedy_decode of library-GEMM logits, on
    exactly representable operands (identical logits, identical hypotheses)."""
    from gluon_e2e_asr_b200 import edit_distance, greedy_decode, proj_greedy_decode
    B, T, K, L = 8, 500, 64, 60
    d = make_batch(B, T, V, L, seed=4)
    th, tw, tb = _exact(B, T, K, V, seed=5, dtype=dtype, dev=dev)
    pl = torch.tensor(d["pred_lengths"], device=dev)
    toks, lens = proj_greedy_decode(th, tw, tb, pl)
    rt, rl = greedy_decode(torch.nn.functional.linear(th.float(), tw.float(), tb), pl, blank=0)
    ref = torch.tensor(d["label"], device=dev).to(torch.int32).contiguous()
    rlen = torch.tensor(d["label_lengths"], device=dev).to(torch.int32).contiguous()
    tot_f = torch.zeros(2, dtype=torch.int64, device=dev)
    tot_r = torch.zeros(2, dtype=torch.int64, device=dev)
    _eq(edit_distance(ref, rlen, toks, lens, tot_f), edit_distance(ref, rlen, rt, rl, tot_r), "per-utterance distances")
    _eq(tot_f, tot_r, "WER totals")
    _eq(toks, rt, "tokens")
    assert int(tot_f[1]) == int(d["label_lengths"].sum()) and int(rl.sum()) > 0
