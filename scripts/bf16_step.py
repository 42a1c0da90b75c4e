"""fp32 against bf16 logits on the device loss path, per BASELINE shape (cfg1-cfg5, tests/synth.py's seeded inputs).

For every shape the fused step (loss + gradient, the ctcb_loss_grad_typed call behind ctc_loss_and_grad) is timed with the
fp32 logits and with the same logits rounded to bf16 -- the bf16 arm gets a bf16 gradient, the fp32 arm an fp32 one.
Raw C-ABI calls (the Python layer's per-call overhead would hide the small shapes), two buffer sets alternating, CUDA
events around windows of back-to-back calls; the two arms alternate window by window in one process, and the spread over
the windows is reported beside the median.  At cfg2 and cfg3 also the forward-only call (ctcb_forward_typed, no history)
and the autograd step (CtcLoss(...)(x, ...).mean().backward(), through Python).  The kernels each arm launched are read
with torch.profiler (a separate, untimed call).  Working sets: cfg3 and cfg5 exceed the 126 MB L2, cfg1/2/4 stay in it
(as in the training loop, which reuses its buffers).

    python scripts/bf16_step.py --out profiles/r5a_bf16_step.json
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gluon_e2e_asr_b200 import CtcLoss, _lib                       # noqa: E402
from gluon_e2e_asr_b200.ops import _Call, _alloc_ws, _stream_ptr   # noqa: E402
from tests.synth import CONFIGS, make_batch                        # noqa: E402

ARMS = (("fp32", torch.float32), ("bf16", torch.bfloat16))


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def make_calls(name, dtype, grad):
    """Two buffer sets of one shape: (callable, kept tensors)."""
    B, T, V, L = CONFIGS[name]
    dev = torch.device("cuda:0")
    lib = _lib.load()
    sets = []
    for i in range(2):
        d = make_batch(B, T, V, L, seed=i)
        x = torch.tensor(d["pred"], device=dev).to(dtype)
        t = [torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths")]
        call = _Call(x, t[0], t[1], t[2], False, True, False)
        loss = torch.empty((B,), device=dev)
        g = torch.empty_like(x) if grad else None
        ws = _alloc_ws(call, grad)
        sets.append((call.problem(loss, g), ws, call.ldt, (x, t, loss, g)))
    st = _stream_ptr(dev)

    def run(i):
        p, ws, ldt = sets[i % 2][:3]
        if grad:
            rc = lib.ctcb_loss_grad_typed(ctypes.byref(p), ldt, ws.data_ptr(), ws.numel(), st)
        else:
            rc = lib.ctcb_forward_typed(ctypes.byref(p), ldt, 0, ws.data_ptr(), ws.numel(), st)
        _lib.check(rc)
    return run, sets


def make_autograd(name, dtype):
    B, T, V, L = CONFIGS[name]
    dev = torch.device("cuda:0")
    d = make_batch(B, T, V, L, seed=0)
    x = torch.tensor(d["pred"], device=dev).to(dtype)
    t = [torch.tensor(d[k], device=dev) for k in ("label", "pred_lengths", "label_lengths")]
    fn = CtcLoss(layout="NTC", label_layout="NT")

    def run(i):
        pred = x.detach().requires_grad_(True)
        fn(pred, *t).mean().backward()
    return run, (x, t)


def kernels_of(run):
    """Kernel names and launch count of one call (profiled, not timed)."""
    run(0)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run(1)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.name.startswith("void ctcb::")]
    return {"launches": _lib.last_launch_count(), "grad_kernel": _lib.last_grad_kernel(),
            "walk_config": list(_lib.last_walk_config()), "kernels": names}


def timed(runs, window_ms, windows):
    """runs: {arm: run(i)}.  Per arm: calls per window sized to ~window_ms, then `windows` windows per arm, alternating."""
    n = {}
    for arm, run in runs.items():
        for i in range(10):
            run(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(20):
            run(i)
        e1.record()
        torch.cuda.synchronize()
        per = e0.elapsed_time(e1) / 20
        n[arm] = max(20, int(window_ms / max(per, 1e-3)))
    res = {arm: [] for arm in runs}
    for w in range(windows):
        for arm, run in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(n[arm]):
                run(i)
            e1.record()
            torch.cuda.synchronize()
            res[arm].append(e0.elapsed_time(e1) / n[arm] * 1e3)
    out = {}
    for arm, v in res.items():
        v = sorted(v)
        out[arm] = {"median_us": round(v[len(v) // 2], 2), "min_us": round(v[0], 2), "max_us": round(v[-1], 2),
                    "calls_per_window": n[arm], "windows": windows}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    ap.add_argument("--window-ms", type=float, default=100.0)
    ap.add_argument("--windows", type=int, default=9)
    ap.add_argument("--shapes", default="cfg1,cfg2,cfg3,cfg4,cfg5")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bf16_step.py measures on the GPU: no CUDA device")
    res = {"what": "per-call device time, us (CUDA events); fp32 and bf16 logits alternating window by window",
           **device_info(), "fused_step": {}, "forward_only": {}, "autograd_step": {}}
    print(json.dumps({k: res[k] for k in ("device", "nvidia_smi")}), flush=True)
    shapes = a.shapes.split(",")
    for name in shapes:
        runs, keep, kern = {}, [], {}
        for arm, dt in ARMS:
            run, sets = make_calls(name, dt, True)
            runs[arm] = run
            keep.append(sets)
            kern[arm] = kernels_of(run)
        r = timed(runs, a.window_ms, a.windows)
        r["kernels"] = kern
        res["fused_step"][name] = r
        print(name, "fused step", json.dumps(r), flush=True)
        del runs, keep
        torch.cuda.empty_cache()
    for name in [s for s in ("cfg2", "cfg3") if s in shapes]:
        runs, keep, kern = {}, [], {}
        for arm, dt in ARMS:
            run, sets = make_calls(name, dt, False)
            runs[arm] = run
            keep.append(sets)
            kern[arm] = kernels_of(run)
        r = timed(runs, a.window_ms, a.windows)
        r["kernels"] = kern
        res["forward_only"][name] = r
        print(name, "forward only", json.dumps(r), flush=True)
        runs, keep = {}, []
        for arm, dt in ARMS:
            run, k = make_autograd(name, dt)
            runs[arm] = run
            keep.append(k)
        r = timed(runs, a.window_ms, a.windows)
        res["autograd_step"][name] = r
        print(name, "autograd step", json.dumps(r), flush=True)
        del runs, keep
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
