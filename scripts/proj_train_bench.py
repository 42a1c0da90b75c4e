"""Times the training call of the output projection fused with the loss -- forward and backward through autograd, d hidden,
d weight and d bias -- at the shape of scripts/proj_bench.py (BASELINE configs[2]: T = 500, V = 2000, L = 150; H = 512
hidden units) for B = 32 / 64 / 128.  Five arms, alternating in one process:

    lib_f32         fused_training=False        library tf32 GEMM writes the logits, CtcLoss forward, k_grad reads them again
    fused_f32       fused_training=True         the fused forward stores the logits, k_grad reads them
    recompute_f32   fused_training="recompute"  no logits: occupancy table in the forward, the product again in the backward
    fused_bf16      fused_training=True         bfloat16 operands (the logits store is forced on this dtype today)
    recompute_bf16  fused_training="recompute"  bfloat16 operands

Every arm ends in the same three contractions (tf32 library GEMMs for d hidden and d weight, the column sum for d bias).
CUDA events on torch's current stream around `iters` steps, inputs resident, L2 flushed by rotating over input sets larger
than L2; `rounds` rounds, the arm order rotated every round.  Per arm: median and [min, max] of the per-round means, and
torch.cuda.max_memory_allocated over one step (beyond the resident inputs).  The GPU's name and power limit are read in
the same run.

    python scripts/proj_train_bench.py [--iters 10 --rounds 7 --out profiles/r5d_proj_train.json] [--profile]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gluon_e2e_asr_b200 import proj_ctc_loss  # noqa: E402
from tests.synth import make_batch  # noqa: E402

ARMS = {"lib_f32": ("f32", False), "fused_f32": ("f32", True), "recompute_f32": ("f32", "recompute"),
        "fused_bf16": ("bf16", True), "recompute_bf16": ("bf16", "recompute")}


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


def bench_batch(a, B, dev):
    sets = []
    for s in range(a.sets):
        d = make_batch(B, a.T, a.V, a.L, seed=s)
        g = torch.Generator(device="cpu").manual_seed(s)
        h = torch.randn((B, a.T, a.H), generator=g).to(dev)
        w = (torch.randn((a.V, a.H), generator=g) / a.H ** 0.5).to(dev)
        sets.append(dict(
            f32=(h.requires_grad_(True), w.requires_grad_(True)),
            bf16=(h.detach().bfloat16().requires_grad_(True), w.detach().bfloat16().requires_grad_(True)),
            bias=torch.zeros((a.V,), device=dev, requires_grad=True),
            lab=torch.tensor(d["label"], device=dev), pl=torch.tensor(d["pred_lengths"], device=dev),
            ll=torch.tensor(d["label_lengths"], device=dev)))

    def step(dt, mode, i):
        s = sets[i % a.sets]
        h, w = s[dt]
        loss = proj_ctc_loss(h, w, s["bias"], s["lab"], s["pl"], s["ll"], fused_training=mode)
        grads = torch.autograd.grad(loss.sum() / B, (h, w, s["bias"]))
        return loss.detach(), grads

    fns = {n: (lambda i, dt=dt, mode=mode: step(dt, mode, i)) for n, (dt, mode) in ARMS.items()}
    out = {}
    # what the arms compute: recompute's losses against fused_training=True's (bit-identical by construction), and its
    # parameter gradients against the logits-store path's
    for dt in ("f32", "bf16"):
        lf, gf = step(dt, True, 0)
        lr, gr = step(dt, "recompute", 0)
        out[dt + "_losses_recompute_equal_fused"] = bool(torch.equal(lf, lr))
        out[dt + "_max_rel_grad_diff_recompute_vs_fused"] = [
            float((x.float() - y.float()).abs().max() / y.float().abs().max()) for x, y in zip(gr, gf)]
    for fn in fns.values():                         # warm-up: module loads, library algorithm choice
        for i in range(3):
            fn(i)
    torch.cuda.synchronize()
    mem = {}
    for n, fn in fns.items():
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        fn(0)
        torch.cuda.synchronize()
        mem[n] = torch.cuda.max_memory_allocated() - base
    names = list(fns)
    per = {n: [] for n in names}
    for r in range(a.rounds):
        for n in names[r % len(names):] + names[:r % len(names)]:
            per[n].append(timed(fns[n], a.iters))
    for n in names:
        v = np.array(per[n])
        out[n] = {"median_us": round(float(np.median(v)), 1), "min_us": round(float(v.min()), 1),
                  "max_us": round(float(v.max()), 1), "rounds_us": [round(float(x), 1) for x in v],
                  "step_peak_bytes_beyond_inputs": int(mem[n])}
    if a.profile:
        out["kernels"] = kernel_times(fns, names)
    return out


def kernel_times(fns, names, steps=5):
    """torch.profiler, a run of its own after the timed rounds: mean device time per step of each kernel, per arm."""
    from torch.profiler import ProfilerActivity, profile
    res = {}
    for n in names:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(steps):
                fns[n](i)
            torch.cuda.synchronize()
        k = {}
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" and e.count > 0:
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                k[e.key[:90]] = round(t / steps, 1)
        res[n] = dict(sorted(k.items(), key=lambda kv: -kv[1]))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, nargs="+", default=[32, 64, 128])
    ap.add_argument("--T", type=int, default=500)
    ap.add_argument("--V", type=int, default=2000)
    ap.add_argument("--L", type=int, default=150)
    ap.add_argument("--H", type=int, default=512)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--sets", type=int, default=2)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", action="store_true", help="also the per-kernel device time of each arm (torch.profiler)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("proj_train_bench.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    res = {"shape": vars(a), "gpu": gpu_info(), "arms": {n: "%s operands, fused_training=%r" % v for n, v in ARMS.items()},
           "timing": "CUDA events around `iters` forward+backward steps per round; per-round means; L2 flushed by rotating "
                     "%d input sets" % a.sets}
    for B in a.B:
        res["B%d" % B] = bench_batch(a, B, dev)
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
