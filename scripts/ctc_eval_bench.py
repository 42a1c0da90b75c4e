"""Times the validation pass over logits -- loss plus greedy hypotheses (train_ctc_ce.py:143-160) -- at the reference's
shapes (BASELINE configs cfg1-cfg5, fp32 logits; cfg2 and cfg3 also with bfloat16 logits).  Four arms, alternating in
one process:

    a  ctc_eval                                   the loss evaluation that also decodes (one read of the logits)
    b  ctc_loss under no_grad, then greedy_decode   the two calls it replaces (two reads)
    c  ctc_loss under no_grad alone                 (a - c: what the decode adds to the loss evaluation)
    d  greedy_decode alone                          (b - c, roughly: what the second read costs)

CUDA events on torch's current stream around `iters` calls per round, `rounds` rounds with the arm order rotated every
round; the median and [min, max] of the per-round means.  The inputs rotate over as many logits sets as it takes to
exceed twice the 126 MB L2 (at most 512 sets), so every call reads its logits from HBM, as a validation loop over a
dev set does.  Before timing, a's outputs are checked against b's bit for bit.  The GPU's name and power limit are read
in the same run.

    python scripts/ctc_eval_bench.py [--iters 100 --rounds 7 --out profiles/r5g_ctc_eval.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gluon_e2e_asr_b200 import ctc_eval, greedy_decode  # noqa: E402
from gluon_e2e_asr_b200.ops import ctc_loss  # noqa: E402
from tests.synth import CONFIGS, make_batch  # noqa: E402

RUNS = [("cfg1", "f32"), ("cfg2", "f32"), ("cfg3", "f32"), ("cfg4", "f32"), ("cfg5", "f32"), ("cfg2", "bf16"), ("cfg3", "bf16")]
L2_BYTES = 126 * 1024 * 1024


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


def bench(cfg, dt, iters, rounds, dev):
    B, T, V, L = CONFIGS[cfg]
    d = make_batch(B, T, V, L, seed=1)
    lab, pl, ll = (torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths"))
    dtype = torch.bfloat16 if dt == "bf16" else torch.float32
    nbytes = B * T * V * (2 if dt == "bf16" else 4)
    nsets = int(min(512, max(2, -(-2 * L2_BYTES // nbytes))))
    g = torch.Generator(device=dev).manual_seed(7)
    xs = [torch.randn((B, T, V), generator=g, device=dev).to(dtype) for _ in range(nsets)]

    def a_eval(i):
        return ctc_eval(xs[i % nsets], lab, pl, ll)

    def b_loss_then_decode(i):
        x = xs[i % nsets]
        with torch.no_grad():
            loss = ctc_loss(x.transpose(0, 1), lab, pl, ll, True, True)
        return (loss,) + greedy_decode(x, pl, blank=0)

    def c_loss(i):
        with torch.no_grad():
            return ctc_loss(xs[i % nsets].transpose(0, 1), lab, pl, ll, True, True)

    def d_decode(i):
        return greedy_decode(xs[i % nsets], pl, blank=0)

    fns = {"a_ctc_eval": a_eval, "b_ctc_loss_then_greedy_decode": b_loss_then_decode, "c_ctc_loss": c_loss,
           "d_greedy_decode": d_decode}
    for i in range(2):                               # what the arms compute: a and b bit for bit
        la, ta, na = a_eval(i)
        lb, tb, nb = b_loss_then_decode(i)
        assert torch.equal(la.view(torch.int32), lb.view(torch.int32)), (cfg, dt, "loss")
        assert torch.equal(ta, tb) and torch.equal(na, nb), (cfg, dt, "hypotheses")
    for fn in fns.values():                          # warm-up: module loads, every set touched once
        for i in range(max(3, nsets)):
            fn(i)
    torch.cuda.synchronize()
    names = list(fns)
    per = {n: [] for n in names}
    for r in range(rounds):
        for n in names[r % len(names):] + names[:r % len(names)]:
            per[n].append(timed(fns[n], iters))
    out = {"B": B, "T": T, "V": V, "Lmax": L, "logits": dt, "input_sets": nsets, "bytes_per_set": nbytes}
    for n in names:
        v = np.array(per[n])
        out[n] = {"median_us": round(float(np.median(v)), 1), "min_us": round(float(v.min()), 1),
                  "max_us": round(float(v.max()), 1)}
    med = {n: out[n]["median_us"] for n in names}
    out["decode_price_a_minus_c_us"] = round(med["a_ctc_eval"] - med["c_ctc_loss"], 1)
    out["saving_b_minus_a_us"] = round(med["b_ctc_loss_then_greedy_decode"] - med["a_ctc_eval"], 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--only", default=None, help="comma-separated cfg:dtype pairs, e.g. cfg2:f32,cfg3:bf16")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ctc_eval_bench.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    runs = [tuple(s.split(":")) for s in a.only.split(",")] if a.only else RUNS
    res = {"gpu": gpu_info(), "iters": a.iters, "rounds": a.rounds,
           "timing": "CUDA events around `iters` calls per round, per-round means: median [min, max]; inputs rotated over "
                     "sets larger than twice L2 together, so the logits are read from HBM"}
    for cfg, dt in runs:
        r = bench(cfg, dt, a.iters, a.rounds, dev)
        res["%s_%s" % (cfg, dt)] = r
        print(json.dumps({"%s_%s" % (cfg, dt): r}), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
