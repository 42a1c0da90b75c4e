"""Times the validation pass -- loss plus greedy hypotheses -- from the encoder output at the shape of
scripts/proj_bench.py (BASELINE configs[2]: B = 64, T = 500, V = 2000, L = 150; H = 512 hidden units).  Four arms
and one breakdown, alternating in one process, for fp32 (tf32 product) and bfloat16 operands:

    a  fused loss only                          proj_ctc_loss under no_grad (the logits never stored)
    b  fused loss + decode                      proj_ctc_eval
    c  library GEMM -> ctc_loss -> greedy_decode  today's way to get both (the logits written once, read twice)
    d  fused loss + library GEMM + greedy_decode
    e  greedy_decode alone on resident logits (the share of c and d that the decode kernel takes)

CUDA events on torch's current stream around `iters` calls, inputs resident, L2 flushed by rotating over buffer sets
larger than L2 (as proj_bench.py does); `rounds` rounds, the arm order rotated every round.  Reports the median and
the spread of the per-round means, and the GPU's name and power limit.

    python scripts/proj_decode_bench.py [--iters 20 --rounds 7 --out profiles/r5b_proj_decode.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gluon_e2e_asr_b200 import greedy_decode, proj_ctc_eval, proj_ctc_loss  # noqa: E402
from gluon_e2e_asr_b200.ops import ctc_loss  # noqa: E402
from tests.synth import make_batch  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = out
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3        # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=64)
    ap.add_argument("--T", type=int, default=500)
    ap.add_argument("--V", type=int, default=2000)
    ap.add_argument("--L", type=int, default=150)
    ap.add_argument("--H", type=int, default=512)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--sets", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("proj_decode_bench.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    sets = []
    for s in range(a.sets):
        d = make_batch(a.B, a.T, a.V, a.L, seed=s)
        g = torch.Generator(device="cpu").manual_seed(s)
        h = torch.randn((a.B, a.T, a.H), generator=g).to(dev)
        w = (torch.randn((a.V, a.H), generator=g) / a.H ** 0.5).to(dev)
        sets.append(dict(
            f32=(h, w), bf16=(h.bfloat16(), w.bfloat16()),
            bias=torch.zeros((a.V,), device=dev),
            lab=torch.tensor(d["label"], device=dev), pl=torch.tensor(d["pred_lengths"], device=dev),
            ll=torch.tensor(d["label_lengths"], device=dev)))
    torch.backends.cuda.matmul.allow_tf32 = True
    res = {"shape": vars(a), "gpu": gpu_info(),
           "timing": "CUDA events around `iters` calls per round; per-round means; L2 flushed by rotating %d input sets" % a.sets}

    def library_logits(s, dt):
        h, w = s[dt]
        if dt == "f32":
            return torch.addmm(s["bias"], h.view(-1, a.H), w.t()).view(a.B, a.T, a.V)
        return (h.view(-1, a.H) @ w.t()).float().add_(s["bias"]).view(a.B, a.T, a.V)

    def arms(dt):
        def fused_loss(i):
            s = sets[i % a.sets]
            with torch.no_grad():
                return proj_ctc_loss(*s[dt], s["bias"], s["lab"], s["pl"], s["ll"])

        def fused_loss_decode(i):
            s = sets[i % a.sets]
            return proj_ctc_eval(*s[dt], s["bias"], s["lab"], s["pl"], s["ll"])

        def gemm_loss_decode(i):
            s = sets[i % a.sets]
            with torch.no_grad():
                logits = library_logits(s, dt)
                loss = ctc_loss(logits.transpose(0, 1), s["lab"], s["pl"], s["ll"], True, True)
                return (loss,) + greedy_decode(logits, s["pl"], blank=0)

        def fused_loss_gemm_decode(i):
            s = sets[i % a.sets]
            with torch.no_grad():
                loss = proj_ctc_loss(*s[dt], s["bias"], s["lab"], s["pl"], s["ll"])
                return (loss,) + greedy_decode(library_logits(s, dt), s["pl"], blank=0)

        with torch.no_grad():
            resident = [library_logits(s, dt) for s in sets]

        def decode_only(i):
            return greedy_decode(resident[i % a.sets], sets[i % a.sets]["pl"], blank=0)

        return {"a_fused_loss": fused_loss, "b_fused_loss_decode": fused_loss_decode,
                "c_gemm_loss_decode": gemm_loss_decode, "d_fused_loss_gemm_decode": fused_loss_gemm_decode,
                "e_greedy_decode_only": decode_only}

    for dt in ("f32", "bf16"):
        fns = arms(dt)
        if dt == "bf16":
            res["bf16_note"] = "the library arms round the logits to bfloat16 (bf16 GEMM output) before widening"
        # what the arms compute: the fused hypotheses against those of the library GEMM's logits (tf32 / bf16 products
        # accumulated in another order: near-ties may flip)
        _, tb, lb = fns["b_fused_loss_decode"](0)
        _, tc, lc = fns["c_gemm_loss_decode"](0)
        same = [(lb[b] == lc[b]).item() and torch.equal(tb[b, :lb[b]], tc[b, :lc[b]]) for b in range(a.B)]
        res[dt + "_identical_hypotheses_fused_vs_library"] = "%d of %d" % (sum(same), a.B)
        for fn in fns.values():                     # warm-up: module loads, library algorithm choice
            for i in range(3):
                fn(i)
        torch.cuda.synchronize()
        names = list(fns)
        per = {n: [] for n in names}
        for r in range(a.rounds):
            for n in names[r % len(names):] + names[:r % len(names)]:
                per[n].append(timed(fns[n], a.iters))
        out = {}
        for n in names:
            v = np.array(per[n])
            out[n] = {"median_us": round(float(np.median(v)), 1), "min_us": round(float(v.min()), 1),
                      "max_us": round(float(v.max()), 1), "rounds_us": [round(float(x), 1) for x in v]}
        med = {n: out[n]["median_us"] for n in names}
        out["decode_price_b_minus_a_us"] = round(med["b_fused_loss_decode"] - med["a_fused_loss"], 1)
        out["b_vs_c_us"] = round(med["b_fused_loss_decode"] - med["c_gemm_loss_decode"], 1)
        out["b_vs_d_us"] = round(med["b_fused_loss_decode"] - med["d_fused_loss_gemm_decode"], 1)
        res[dt] = out
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
