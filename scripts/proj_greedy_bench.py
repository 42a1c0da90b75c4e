"""Times the label-free greedy decode from the encoder output (decode_ctc.py:118-140) at the shape of
scripts/proj_bench.py (BASELINE configs[2]: B = 64, T = 500, V = 2000, L = 150; H = 512 hidden units, variable lengths),
for fp32 (tf32 product) and bfloat16 operands, arms alternating in one process:

    a  proj_greedy_decode                         the projection's decode-only epilogue + the collapse kernel
    b  library GEMM -> greedy_decode              the decode script's way until now (the logits written, then read)
    c  proj_ctc_eval                              loss + decode epilogue, walkers, collapse (the validation pass)
    d  fused loss only                            proj_ctc_loss under no_grad
    e  proj_greedy_decode with proj_dbg=1         the epilogue skips its arithmetic (results garbage): the projection's
                                                  TMA + MMA time and the collapse launch -- the floor under a

and one small-vocabulary shape (V = 46, B = 32, T = 500, H = 512) with arms a and b.  Before timing, a's tokens and
lengths are asserted equal to c's.  CUDA events on torch's current stream around `iters` calls, inputs resident, L2
flushed by rotating over input sets larger than L2; `rounds` rounds, the arm order rotated every round.  Reports the
median and [min, max] of the per-round means, and the GPU's name and power limit, read in the same run.

    python scripts/proj_greedy_bench.py [--iters 20 --rounds 7 --out profiles/r5c_proj_greedy.json]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gluon_e2e_asr_b200 import _lib, greedy_decode, proj_ctc_eval, proj_ctc_loss, proj_greedy_decode  # noqa: E402
from scripts.proj_decode_bench import gpu_info, timed  # noqa: E402
from tests.synth import make_batch  # noqa: E402


def make_sets(B, T, V, L, H, n, dev):
    sets = []
    for s in range(n):
        d = make_batch(B, T, V, L, seed=s)
        g = torch.Generator(device="cpu").manual_seed(s)
        h = torch.randn((B, T, H), generator=g).to(dev)
        w = (torch.randn((V, H), generator=g) / H ** 0.5).to(dev)
        sets.append(dict(f32=(h, w), bf16=(h.bfloat16(), w.bfloat16()), bias=(torch.randn((V,), generator=g) * 0.5).to(dev),
                         lab=torch.tensor(d["label"], device=dev), pl=torch.tensor(d["pred_lengths"], device=dev),
                         ll=torch.tensor(d["label_lengths"], device=dev)))
    return sets


def library_logits(s, dt):
    h, w = s[dt]
    B, T, H = h.shape
    if dt == "f32":
        return torch.addmm(s["bias"], h.view(-1, H), w.t()).view(B, T, -1)
    return (h.view(-1, H) @ w.t()).float().add_(s["bias"]).view(B, T, -1)


def run_arms(fns, rounds, iters):
    for fn in fns.values():                     # warm-up: module loads, library algorithm choice
        for i in range(3):
            fn(i)
    torch.cuda.synchronize()
    names = list(fns)
    per = {n: [] for n in names}
    for r in range(rounds):
        for n in names[r % len(names):] + names[:r % len(names)]:
            per[n].append(timed(fns[n], iters))
    out = {}
    for n in names:
        v = np.array(per[n])
        out[n] = {"median_us": round(float(np.median(v)), 1), "min_us": round(float(v.min()), 1),
                  "max_us": round(float(v.max()), 1), "rounds_us": [round(float(x), 1) for x in v]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=64)
    ap.add_argument("--T", type=int, default=500)
    ap.add_argument("--V", type=int, default=2000)
    ap.add_argument("--L", type=int, default=150)
    ap.add_argument("--H", type=int, default=512)
    ap.add_argument("--small-B", type=int, default=32)
    ap.add_argument("--small-V", type=int, default=46)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--sets", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("proj_greedy_bench.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    torch.backends.cuda.matmul.allow_tf32 = True
    res = {"shape": vars(a), "gpu": gpu_info(),
           "timing": "CUDA events around `iters` calls per round; per-round means; L2 flushed by rotating %d input sets" % a.sets,
           "bf16_note": "the library arm rounds the logits to bfloat16 (bf16 GEMM output) before widening"}

    sets = make_sets(a.B, a.T, a.V, a.L, a.H, a.sets, dev)
    for dt in ("f32", "bf16"):
        def greedy(i, dt=dt):
            s = sets[i % a.sets]
            return proj_greedy_decode(*s[dt], s["bias"], s["pl"])

        def gemm_greedy(i, dt=dt):
            s = sets[i % a.sets]
            with torch.no_grad():
                return greedy_decode(library_logits(s, dt), s["pl"], blank=0)

        def evaluate(i, dt=dt):
            s = sets[i % a.sets]
            return proj_ctc_eval(*s[dt], s["bias"], s["lab"], s["pl"], s["ll"])

        def fused_loss(i, dt=dt):
            s = sets[i % a.sets]
            with torch.no_grad():
                return proj_ctc_loss(*s[dt], s["bias"], s["lab"], s["pl"], s["ll"])

        def floor(i, dt=dt):
            with _lib.options(proj_dbg=1):
                return greedy(i)

        for k in range(a.sets):                 # what a computes: proj_ctc_eval's hypotheses, bit for bit
            ta, la = greedy(k)
            _, tc, lc = evaluate(k)
            assert torch.equal(ta, tc) and torch.equal(la, lc), "proj_greedy_decode differs from proj_ctc_eval (%s)" % dt
        tb, lb = gemm_greedy(0)
        same = [(la[b] == lb[b]).item() and torch.equal(ta[b, :la[b]], tb[b, :lb[b]]) for b in range(a.B)]
        out = run_arms({"a_proj_greedy_decode": greedy, "b_gemm_greedy_decode": gemm_greedy, "c_proj_ctc_eval": evaluate,
                        "d_fused_loss": fused_loss, "e_greedy_epilogue_skipped": floor}, a.rounds, a.iters)
        med = {n: v["median_us"] for n, v in out.items()}
        out["a_equals_c"] = True
        out["identical_hypotheses_a_vs_b"] = "%d of %d" % (sum(same), a.B)
        out["b_minus_a_us"] = round(med["b_gemm_greedy_decode"] - med["a_proj_greedy_decode"], 1)
        out["c_minus_a_us"] = round(med["c_proj_ctc_eval"] - med["a_proj_greedy_decode"], 1)
        out["a_minus_d_us"] = round(med["a_proj_greedy_decode"] - med["d_fused_loss"], 1)
        out["epilogue_price_a_minus_e_us"] = round(med["a_proj_greedy_decode"] - med["e_greedy_epilogue_skipped"], 1)
        res[dt] = out

    small = make_sets(a.small_B, a.T, a.small_V, 60, a.H, a.sets, dev)
    res["small_shape"] = {"B": a.small_B, "T": a.T, "V": a.small_V, "H": a.H}
    for dt in ("f32", "bf16"):
        def greedy(i, dt=dt):
            s = small[i % a.sets]
            return proj_greedy_decode(*s[dt], s["bias"], s["pl"])

        def gemm_greedy(i, dt=dt):
            s = small[i % a.sets]
            with torch.no_grad():
                return greedy_decode(library_logits(s, dt), s["pl"], blank=0)

        ta, la = greedy(0)
        tb, lb = gemm_greedy(0)
        same = [(la[b] == lb[b]).item() and torch.equal(ta[b, :la[b]], tb[b, :lb[b]]) for b in range(a.small_B)]
        out = run_arms({"a_proj_greedy_decode": greedy, "b_gemm_greedy_decode": gemm_greedy}, a.rounds, a.iters)
        out["identical_hypotheses_a_vs_b"] = "%d of %d" % (sum(same), a.small_B)
        res["small_" + dt] = out
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
