#!/usr/bin/env python
"""bench.py -- CTC fwd+bwd valid frames/s on B200 (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfgX] [--impl reference] [--dump-outputs DIR]

A *step* is one pass of the hot path (log-softmax, alpha/beta recursion, gradient to the logits) over one
synthetic batch.

Workloads (BASELINE.json `configs`):
  N = 1  -> configs[1], cfg2: B=32, T=500, V=46, L<=120, variable lengths (the headline).  The same run also
            measures the other configs as context (`other_workloads`), cfg5 -- the N=1 point of the
            sharded sweep -- among them (`sweep`).
  N > 1  -> configs[4], cfg5: ONE batch of B=1024 (T=500, V=46, L=120, full lengths) split by utterance over
            the N ranks with the reference's own split (scripts/swbd/utils.py:25-33 `split_and_load`,
            gluon_e2e_asr_b200.sharding.shard_for_rank), "scaling": "strong".  No data-path collective; the
            float64 loss sum of every step is exchanged over NVLink (peer mailbox, or --collective nccl).
            Rank 0 also times the WHOLE batch alone on its GPU in the same run (`sweep.single_gpu_ms`).

`value`  : device-resident inputs, the step's kernels (and the exchange) replayed from CUDA graphs, CUDA events
           around exactly K steps behind a device-side start gate, max over ranks.
`e2e`    : the same metric through the drop-in boundary with HOST buffers: the C ABI's prefetching host entry
           (ctcb_pipe_submit / ctcb_pipe_wait) with pinned host batches -- every step's H2D of
           logits/labels/lengths, its kernels and the D2H of its loss vector are inside the timed loop and every
           loss is read on the host; batch i+1's copy overlaps batch i's kernels; the gradient stays on the
           device, where the model's backward consumes it.  At N > 1 every step also all-reduces its loss sum.
`e2e_sync` / `e2e_plugin`: the synchronous host entry, and the Python mirror of the reference's block
           (CtcLoss(...)(pred, ...).mean().backward(), torch autograd on the path) -- N = 1 only.
`roofline`: dominant kernel against the measured HBM copy peak; `traffic` = whole-step DRAM bytes from
           profiles/traffic.json (written by scripts/make_traffic.py from an ncu --cache-control none capture).
`cpu_baseline`: the oracle's C restatement of the reference's CPU operator on this box's host cores (all
           cores and one thread), torch's CPU ctc_loss as an independent second number and an `import mxnet`
           probe (N = 1, rank 0 only; bounded samples).
`--impl reference`: the same C restatement as the measured arm (the reference's MXNet operator is not
           installable here -- DESIGN.md section 2), all host threads, SAME workload, seeds and config keys.
`--dump-outputs DIR`: after the K timed steps, the outputs of the last one -- per-utterance losses `loss.npy` and
           the logit gradient `grad.npy`, float32 -- go to DIR (one rank only).  The gradient is written whole when
           it fits 63 MB, otherwise as a fixed seeded sample of utterances; `grad_rows.npy` lists which.  The inputs
           depend only on the arguments, so two builds can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

from tests.synth import CONFIGS, make_batch

METRIC = "ctc_fwd_bwd_valid_frames_per_sec"
UNIT = "frames/s"
L2_BYTES = 126 * 1024 * 1024


def algorithmic_bytes(V, T, B, Tb, Lb):
    """SURVEY.md 8(d): read valid logits once + write the dense gradient once + labels/lengths/loss."""
    return 4 * V * int(Tb.sum()) + 4 * V * B * T + 4 * int(Lb.sum()) + 12 * B


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------
# the workload, shared by both arms: same shapes, same seeds, same config keys
# ------------------------------------------------------------------------------------------
def default_workload(world):
    return "cfg2" if world == 1 else "cfg5"


def n_sets(name):
    """Distinct input sets the timed loop rotates over: enough (logits + gradient) bytes to exceed L2."""
    B, T, V, L = CONFIGS[name]
    per_set = 2 * 4 * B * T * V
    n = max(2, min(64, (2 * L2_BYTES + per_set - 1) // per_set + 1))
    return n - (n % 2)


def batch_for(name, i):
    """Input set i of the rotation: seed = i (both arms)."""
    B, T, V, L = CONFIGS[name]
    return make_batch(B, T, V, L, seed=i, full_lengths=(name == "cfg5"))


def workload_config(name, world, steps, frames_per_step):
    B, T, V, L = CONFIGS[name]
    return {
        "workload": name, "B": B, "T": T, "V": V, "Lmax": L, "layout": "NTC",
        "lengths": "full" if name == "cfg5" else "variable",
        "seeds": "set i of the rotation = tests.synth.make_batch(seed=i), %d sets" % n_sets(name),
        "valid_frames_per_step": frames_per_step,
        "sharding": ("none" if world == 1 else
                     "utterances split over %d ranks by the reference's split_and_load (utils.py:25-33)" % world),
    }


def frames_per_step(name, steps, frames_of_set):
    n = n_sets(name)
    return sum(frames_of_set[i % n] for i in range(steps)) / float(steps)


DUMP_GRAD_BYTES = 63 * 10 ** 6      # the gradient's share of the 64 MB a dump may take; losses and row indices are small


def dump_outputs(out_dir, loss, grad):
    """Writes one step's outputs as float32 .npy files: loss (B,), grad (rows, T, V) and grad_rows, the utterance of
    every gradient row -- all of them when the gradient fits DUMP_GRAD_BYTES, else a sample drawn with a fixed seed."""
    B = grad.shape[0]
    n = min(B, DUMP_GRAD_BYTES // (4 * grad[0].size))
    rows = np.arange(B) if n == B else np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for key, a in (("loss", loss), ("grad", grad[rows]), ("grad_rows", rows)):
        np.save(os.path.join(out_dir, key + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


class ClockSampler(threading.Thread):
    """NVML samples of SM clock and throttle reasons while the timed region runs."""

    def __init__(self, index, period=0.004):
        super().__init__(daemon=True)
        self.period, self.samples, self.reasons, self.max_mhz = period, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def sample(self):
        if not self.ok:
            return
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
                     0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}
            for bit, n in names.items():
                if r & bit:
                    self.reasons.add(n)
        except Exception:
            pass

    def run(self):
        while not self._stop_evt.is_set():
            self.sample()
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=1.0)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle's C restatement on the host cores
# ------------------------------------------------------------------------------------------
def host_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_step_fn(d, threads=None):
    from oracle import ctc_ref
    B = d["pred"].shape[0]
    head = np.full((B,), 1.0 / B, np.float32)
    g = np.empty_like(d["pred"])
    lab = d["label"].astype(np.int32)
    # all host threads this process may use (torchrun exports OMP_NUM_THREADS=1: ask explicitly)
    cores = min(host_cores(), B) if threads is None else threads

    def step():
        # NTC logits addressed through strides (no swapaxes copy: a favour to the baseline),
        # softmax + alpha + beta + grad + head scaling, OpenMP over the minibatch
        return ctc_ref.ctc_ref(d["pred"], lab, d["pred_lengths"], d["label_lengths"], blank=0, head_grad=head,
                               layout="NTC", dtype=np.float32, out_grad=g, num_threads=cores)
    return step, cores


def time_cpu_rotation(name, steps, warmup, budget_s=None, threads=None):
    """`steps` CPU steps over the same rotation of input sets the CUDA arm uses; returns (seconds per step list,
    frames per step list, cores, (loss, grad, feasible) of the last step)."""
    n = n_sets(name)
    sets, fns = {}, {}

    def fn(i):
        k = i % n
        if k not in fns:
            sets[k] = batch_for(name, k)
            fns[k] = cpu_step_fn(sets[k], threads)
        return fns[k][0], float(sets[k]["pred_lengths"].sum()), fns[k][1]
    for i in range(warmup):
        fn(i)[0]()
    ts, fr, cores, out = [], [], 1, None
    t_start = time.perf_counter()
    for i in range(steps):
        f, frames, cores = fn(i)
        t0 = time.perf_counter()
        out = f()
        ts.append(time.perf_counter() - t0)
        fr.append(frames)
        if budget_s is not None and time.perf_counter() - t_start > budget_s and len(ts) >= 3:
            break
    return ts, fr, cores, out


def run_reference(args, rank, world):
    if rank != 0:
        return
    name = args.workload or default_workload(world)
    B, T, V, L = CONFIGS[name]
    warm = max(args.warmup, 1)
    ts, fr, cores, last = time_cpu_rotation(name, args.steps, min(warm, 3))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last[0], last[1])
    ms = 1e3 * sum(ts) / len(ts)
    val = sum(fr) / sum(ts)
    n = n_sets(name)
    fos = {i: float(batch_for(name, i)["pred_lengths"].sum()) for i in range(min(n, args.steps))}
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(ts), "warmup": warm, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, world, args.steps, frames_per_step(name, args.steps, fos)),
        "impl_notes": {"what": "C restatement of the reference's CPU CTC operator (oracle/ctc_ref.c, fp32, OpenMP over the "
                               "minibatch: the parallelisation MXNet's CPU operator uses); MXNet itself is not installable in "
                               "this image; the whole batch on this box's host cores, whatever N"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d full %s steps (B=%d)" % (len(ts), name, B)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def extra_cpu_baselines(d, name):
    """One thread of the C port, torch's CPU ctc_loss, and the MXNet probe (SURVEY 8c/8d, BASELINE.md section 3)."""
    out = {}
    frames = float(d["pred_lengths"].sum())
    try:
        step, _ = cpu_step_fn(d, threads=1)
        step()
        ts = []
        t_start = time.perf_counter()
        while len(ts) < 3 or (time.perf_counter() - t_start < 4.0 and len(ts) < 50):
            t0 = time.perf_counter(); step(); ts.append(time.perf_counter() - t0)
        out["one_thread"] = {"value": frames / statistics.median(ts), "unit": UNIT, "cores": 1, "kind": "port",
                             "ms_per_step": 1e3 * statistics.median(ts), "sample": "%d full %s steps" % (len(ts), name)}
    except Exception as exc:  # noqa: BLE001
        out["one_thread"] = {"error": str(exc)[:160]}
    try:
        import torch
        import torch.nn.functional as F
        cores = min(host_cores(), 64)
        old = torch.get_num_threads()
        torch.set_num_threads(cores)
        x = torch.tensor(d["pred"], requires_grad=True)
        lab = torch.tensor(d["label"]).long()
        tl = torch.tensor(d["pred_lengths"]).long(); ll = torch.tensor(d["label_lengths"]).long()

        def tstep():
            x.grad = None
            lp = F.log_softmax(x.transpose(0, 1), dim=2)
            F.ctc_loss(lp, lab, tl, ll, blank=0, reduction="none", zero_infinity=False).mean().backward()
        tstep()
        ts = []
        t_start = time.perf_counter()
        while len(ts) < 3 or (time.perf_counter() - t_start < 4.0 and len(ts) < 50):
            t0 = time.perf_counter(); tstep(); ts.append(time.perf_counter() - t0)
        torch.set_num_threads(old)
        out["torch_cpu"] = {"value": frames / statistics.median(ts), "unit": UNIT, "cores": cores, "kind": "torch F.ctc_loss(log_softmax) fp32 + backward",
                            "ms_per_step": 1e3 * statistics.median(ts), "sample": "%d full %s steps" % (len(ts), name)}
    except Exception as exc:  # noqa: BLE001
        out["torch_cpu"] = {"error": str(exc)[:160]}
    try:
        import mxnet as mx  # noqa: F401  -- the reference's own operator, if a box ever has it
        out["mxnet_probe"] = "import mxnet succeeded (version %s): run tests/golden/make_golden.py --mxnet to pin the oracle" % mx.__version__
    except Exception as exc:  # noqa: BLE001
        out["mxnet_probe"] = "absent (%s: %s) -- parity stays unpinned by the reference itself" % (type(exc).__name__, str(exc)[:80])
    return out


# ------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------
def run_cuda(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from gluon_e2e_asr_b200 import CtcLoss, _lib
    from gluon_e2e_asr_b200 import ops
    from gluon_e2e_asr_b200.sharding import shard_for_rank

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device and no CPU fallback for the measured arm")
    lib = _lib.load()
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # NVML is initialised by every rank BEFORE anything is timed (N processes contend for it)
    sampler = ClockSampler(local_rank if "CUDA_VISIBLE_DEVICES" not in os.environ else 0)

    name = args.workload or default_workload(world)
    Bg, T, V, L = CONFIGS[name]
    sl = shard_for_rank(Bg, rank, world)                       # this rank's utterances (the reference's contiguous split)
    B = sl.stop - sl.start
    nset = n_sets(name)
    per_set = 2 * 4 * B * T * V
    head_g = torch.full((Bg,), 1.0 / Bg, device=dev)           # .mean() over the WHOLE batch (train_ctc_ce.py:363-366)
    head = head_g[sl]

    def to_dev(d, s):
        return {"np": {k: v[s] for k, v in d.items()},
                "pred": torch.tensor(d["pred"][s], device=dev), "label": torch.tensor(d["label"][s], device=dev),
                "pl": torch.tensor(d["pred_lengths"][s], device=dev), "ll": torch.tensor(d["label_lengths"][s], device=dev),
                "loss": torch.empty((s.stop - s.start,), device=dev),
                "grad": torch.empty((s.stop - s.start, T, V), device=dev),
                "frames": float(d["pred_lengths"][s].sum())}
    sets, frames_global, full0 = [], {}, None
    for i in range(nset):
        d = batch_for(name, i)
        frames_global[i] = float(d["pred_lengths"].sum())
        sets.append(to_dev(d, sl))
        if i == 0 and world > 1:
            full0 = d
    # Per-step loss sum (float64, accumulated by the walkers) and its exchange.  Two slots: step i accumulates into
    # slot i % 2 while the exchange inside the same step's graph handles slot (i-1) % 2 -- the previous step's sum.
    part = torch.zeros((2, 3), dtype=torch.float64, device=dev)         # per slot: partial {loss sum, frames, utterances}
    loss_sums = part[:, 0]
    red_buf = torch.zeros((2, 3), dtype=torch.float64, device=dev)
    exchange = world > 1 and not args.no_allreduce

    def step_eager(s, slot=0, hd=None):
        ops.ctc_loss_and_grad(s["pred"], s["label"], s["pl"], s["ll"], head_grad=head if hd is None else hd,
                              loss_sum=loss_sums[slot], out_loss=s["loss"], out_grad=s["grad"], handoff="pointer")

    peer, collective = None, "none"
    if exchange:
        collective = "nccl"
        if args.collective == "peer":
            try:
                from gluon_e2e_asr_b200 import PeerLossSum
                peer = PeerLossSum(dev, lag=args.peer_lag)
                collective = "peer"
            except Exception as exc:  # noqa: BLE001
                if rank == 0:
                    print("bench.py: peer mailbox unavailable (%s); using the NCCL all-reduce" % str(exc)[:160], file=sys.stderr)

    def reduce_slot(slot):
        if peer is not None:
            peer.exchange(part[slot], red_buf[slot])
        else:
            red_buf[slot].copy_(part[slot], non_blocking=True)
            part[slot].zero_()
            dist.all_reduce(red_buf[slot])

    stream = torch.cuda.Stream(dev)
    comm_stream = torch.cuda.Stream(dev)
    graphs = []
    with torch.cuda.stream(stream):
        for i, s in enumerate(sets[:2]):
            step_eager(s, i % 2)
        launches_per_step = _lib.last_launch_count()
        if exchange:
            reduce_slot(0); reduce_slot(1)              # warm-up of the exchange outside any capture (same count on every rank)
        torch.cuda.synchronize()
        walk_cfg = _lib.last_walk_config()
        for i, s in enumerate(sets):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                if exchange and peer is not None:
                    # the previous step's slot: a one-warp kernel behind the step's gradient kernel, as its programmatic dependent
                    peer.exchange_with_next(part[(i + 1) % 2], red_buf[(i + 1) % 2])
                elif exchange:
                    comm_stream.wait_stream(stream)
                    with torch.cuda.stream(comm_stream):
                        reduce_slot((i + 1) % 2)        # the previous step's slot, on a side branch of the graph
                step_eager(s, i % 2)
                if exchange and peer is None:
                    stream.wait_stream(comm_stream)
            graphs.append(g)
    torch.cuda.synchronize()

    # ---- sharded results == single-GPU results (N > 1): the shard's losses carry the bits of the whole batch's ----
    shard_check = None
    if world > 1:
        mine = sets[0]["loss"].clone()
        gathered = [torch.empty((s.stop - s.start,), device=dev) for s in [shard_for_rank(Bg, r, world) for r in range(world)]]
        dist.all_gather(gathered, mine)
        if rank == 0:
            whole = to_dev(full0, slice(0, Bg))
            ops.ctc_loss_and_grad(whole["pred"], whole["label"], whole["pl"], whole["ll"], head_grad=head_g,
                                  out_loss=whole["loss"], out_grad=whole["grad"], handoff="pointer")
            torch.cuda.synchronize()
            same = torch.equal(torch.cat(gathered), whole["loss"])
            gd = (whole["grad"][sl] - sets[0]["grad"]).abs().max().item()
            shard_check = {"per_utterance_losses_bit_identical_to_single_gpu": bool(same), "max_abs_grad_difference_rank0_shard": gd}
            if not same:
                raise SystemExit("bench.py: sharded losses differ from the single-GPU losses")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    gate = torch.zeros((1,), device=dev)

    def run_steps(k, graph=True):
        with torch.cuda.stream(stream):
            for i in range(k):
                if graph:
                    graphs[i % nset].replay()
                else:
                    step_eager(sets[i % nset], i % 2)

    # ---- value: K steps, device-resident inputs ------------------------------------------------
    # Start gate: after the host barrier every rank enqueues one un-timed all-reduce on the timed stream and records
    # its start event right behind it -- the collective ends on all ranks together, so the timed regions start together
    # on the DEVICES whatever the skew between the host processes.
    # One rank: the step's launch mechanism is chosen by an un-timed calibration -- per-step CUDA graphs, or eager launches,
    # where the recursion kernel of step i+1 is the programmatic dependent of step i's gradient kernel (its CTAs become
    # resident during that kernel's tail and wait there: option walk_pdl), which a chain of separate graph launches cannot have.
    use_graph, calib = True, None
    if world == 1:
        def quick(g_):
            run_steps(3, g_)
            torch.cuda.synchronize()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record(stream)
            run_steps(30, g_)
            q1.record(stream)
            torch.cuda.synchronize()
            return q0.elapsed_time(q1) / 30
        calib = {"graph_ms_per_step": quick(True), "eager_ms_per_step": quick(False)}
        use_graph = calib["graph_ms_per_step"] <= calib["eager_ms_per_step"]
    barrier()
    run_steps(args.warmup, use_graph)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    with torch.cuda.stream(stream):
        if world > 1:
            dist.all_reduce(gate)
        elif args.start_gate_us > 0:
            # one rank: a hold kernel ahead of the start event -- the host queues the event and the first steps behind it, so
            # the clock starts with work already in the stream (what the all-reduce gate does at N > 1).  Without it the K
            # timed steps carry the host's launch latency of the first one: a fixed cost of about one and a half steps that a
            # 20-step region shows (49.6 us per step) and a 2000-step region does not (46.0)
            torch.cuda._sleep(int(args.start_gate_us * 1e-6 * 1.9e9))       # cycles at ~1.9 GHz
        e0.record(stream)
    run_steps(args.steps, use_graph)
    e1.record(stream)
    sampler.sample()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    if args.dump_outputs:
        last = sets[(args.steps - 1) % nset]
        dump_outputs(args.dump_outputs, last["loss"].cpu().numpy(), last["grad"].cpu().numpy())
    barrier()
    ms_total = e0.elapsed_time(e1)
    frames_all = sum(frames_global[i % nset] for i in range(args.steps))
    if world > 1:
        tmax = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms_total = tmax[0].item()
    value = frames_all / (ms_total * 1e-3)
    ms_per_step = ms_total / args.steps

    # eager (no CUDA graph) timing of the same steps without the exchange, for the record
    barrier()
    ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    run_steps(min(args.warmup, 5), graph=False)
    ee0.record(stream)
    n_eager = min(args.steps, 200)
    run_steps(n_eager, graph=False)
    ee1.record(stream)
    torch.cuda.synchronize()
    eager_ms = ee0.elapsed_time(ee1) / n_eager

    # ---- the sweep's single-GPU point, same box, same run: rank 0 alone takes the WHOLE batch (N > 1) ----
    sweep = None
    if world > 1:
        single_ms = None
        if rank == 0:
            wsets = [to_dev(batch_for(name, i), slice(0, Bg)) for i in range(nset)]
            k1 = max(5, min(args.steps, 50))
            with torch.cuda.stream(stream):
                for i in range(3):
                    step_eager(wsets[i % nset], 0, head_g)
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record(stream)
                for i in range(k1):
                    step_eager(wsets[i % nset], 0, head_g)
                s1.record(stream)
            torch.cuda.synchronize()
            single_ms = s0.elapsed_time(s1) / k1
            del wsets
            for k in [k for k in ops._ws_cache if k[3] == Bg]:        # the whole-batch workspace only: the graphs hold the shard's
                del ops._ws_cache[k]
            torch.cuda.empty_cache()
        barrier()
        sweep = {"workload": "%s: one B=%d batch split by utterance" % (name, Bg), "n_gpus": world,
                 "ms_per_step": ms_per_step, "value": value, "unit": UNIT,
                 "single_gpu_ms_per_step_same_batch_same_box": single_ms,
                 "utterances_per_rank": B, "shard_check": shard_check}

    # ---- e2e ---------------------------------------------------------------------------------
    from gluon_e2e_asr_b200.batch import PinnedBatch
    import gc
    hsets = []
    for s in sets[:min(nset, 8)]:
        d = s["np"]
        hsets.append(PinnedBatch.from_arrays(np.ascontiguousarray(d["pred"]), np.ascontiguousarray(d["label"]),
                                             np.ascontiguousarray(d["pred_lengths"]), np.ascontiguousarray(d["label_lengths"])))
    loss_host = torch.empty((B,), dtype=torch.float32).pin_memory()
    d2h = int(loss_host.numel() * 4)
    gc.collect()
    gc.freeze()        # the bench holds thousands of long-lived objects (input sets, graphs): keep the collector off them
    e2e_steps = max(10, min(args.steps, 200))
    probs = []
    for h in hsets:
        q = _lib.Problem()
        q.T, q.B, q.V, q.Lmax, q.blank, q.label_pad = T, B, V, L, 0, 0
        q.logits, q.logits_stride_t, q.logits_stride_b = h.pred.data_ptr(), V, T * V
        q.labels, q.label_dtype, q.label_stride_b, q.label_stride_l = h.label.data_ptr(), _lib.DT_F32, L, 1
        q.data_lengths, q.data_lengths_dtype = h.pred_lengths.data_ptr(), _lib.DT_F32
        q.label_lengths, q.label_lengths_dtype = h.label_lengths.data_ptr(), _lib.DT_F32
        q.loss = loss_host.data_ptr()
        probs.append(q)
    hframes = [s["frames"] for s in sets[:len(hsets)]]

    e2e_plugin = e2e_cabi = None
    if world == 1:
        # (a) the Python mirror of the reference's block + torch autograd
        blk = CtcLoss(layout="NTC", label_layout="NT")
        for h in hsets:
            h.load(dev)["pred"].requires_grad_(True)

        def plugin_step(h):
            x = h.load(dev)                                 # one cudaMemcpyAsync: logits, labels, both length vectors
            pred = x["pred"]
            pred.grad = None
            loss = blk(pred, x["label"], x["pred_lengths"], x["label_lengths"])
            loss.mean().backward()
            loss_host.copy_(loss.detach(), non_blocking=True)
            torch.cuda.current_stream().synchronize()       # the step's result is on the host
        for i in range(max(3, min(args.warmup, 10))):
            plugin_step(hsets[i % len(hsets)])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            plugin_step(hsets[i % len(hsets)])
        pm = (time.perf_counter() - t0) * 1e3
        pf = sum(hframes[i % len(hsets)] for i in range(e2e_steps))
        e2e_plugin = {"value": pf / (pm * 1e-3), "unit": UNIT, "h2d_bytes_per_step": hsets[0].h2d_bytes, "d2h_bytes_per_step": d2h,
                      "ms_per_step": pm / e2e_steps, "steps": e2e_steps,
                      "api": "PinnedBatch.load(dev) -> CtcLoss(layout='NTC',label_layout='NT')(pred,label,pred_lengths,"
                             "label_lengths).mean().backward() -> loss to pinned host (torch autograd on the path)"}
        # (b) the C ABI's synchronous host entry
        try:
            dgrad = ctypes.c_void_p()
            for i in range(5):
                _lib.check(lib.ctcb_loss_grad_host_resident(ctypes.byref(probs[i % len(probs)]), local_rank, ctypes.byref(dgrad)))
            t0 = time.perf_counter()
            for i in range(e2e_steps):
                _lib.check(lib.ctcb_loss_grad_host_resident(ctypes.byref(probs[i % len(probs)]), local_rank, ctypes.byref(dgrad)))
            cm = (time.perf_counter() - t0) * 1e3
            e2e_cabi = {"value": pf / (cm * 1e-3), "unit": UNIT, "ms_per_step": cm / e2e_steps,
                        "h2d_bytes_per_step": sum(int(getattr(hsets[0], k).numel() * getattr(hsets[0], k).element_size()) for k in PinnedBatch.FIELDS),
                        "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                        "api": "ctcb_loss_grad_host_resident(problem with pinned HOST pointers): H2D, kernels, loss back to the "
                               "host, gradient left on the device; host wall clock around the synchronous calls"}
        except Exception as exc:  # noqa: BLE001
            e2e_cabi = {"error": str(exc)[:200]}

    # (c) the C ABI's prefetching host entry (the headline): batch i+1's H2D in flight while batch i's kernels run; every
    # step's loss (and loss sum) is read on the host before the step counts; at N > 1 the loss sums of every step are
    # all-reduced over the ranks (NCCL) before the step counts -- the reference's per-step `+=` over the shards
    # (train_ctc_ce.py:367-368)
    e2e_pipe = None
    try:
        depth = args.pipe_depth
        ph = ctypes.c_void_p()
        _lib.check(lib.ctcb_pipe_create(local_rank, depth, ctypes.byref(ph)))
        loss_bufs = [torch.zeros((B,), dtype=torch.float32).pin_memory() for _ in hsets]
        sum_bufs = [torch.zeros((1,), dtype=torch.float64).pin_memory() for _ in hsets]
        loss_np = [b.numpy() for b in loss_bufs]
        # the pipe's batches are PACKED on the host (PinnedBatch(packed=True), ctcb_problem_t.logits_row_offsets): the
        # collation writes only the valid frames of every utterance, so the padded frames never cross PCIe
        psets = []
        for s_ in sets[:len(hsets)]:
            d = s_["np"]
            psets.append(PinnedBatch.from_arrays(np.ascontiguousarray(d["pred"]), np.ascontiguousarray(d["label"]),
                                                 np.ascontiguousarray(d["pred_lengths"]), np.ascontiguousarray(d["label_lengths"]),
                                                 packed=not args.dense_host))
        pprobs = []
        for q0, pk, lb, sb in zip(probs, psets, loss_bufs, sum_bufs):
            q = _lib.Problem()
            ctypes.memmove(ctypes.byref(q), ctypes.byref(q0), ctypes.sizeof(q))
            q.logits = pk.pred.data_ptr()
            q.labels = pk.label.data_ptr()
            q.data_lengths, q.label_lengths = pk.pred_lengths.data_ptr(), pk.label_lengths.data_ptr()
            if pk.packed:
                q.logits_row_offsets = pk.row_offsets.data_ptr()
            q.loss = lb.data_ptr()
            if world > 1:
                q.loss_sum = sb.data_ptr()              # the shard's float64 loss sum, for the all-reduce over the ranks
            pprobs.append(q)
        npb = len(pprobs)
        tk = ctypes.c_int64(-1)
        moved = {}
        hb, pulled = ctypes.c_int64(0), ctypes.c_int32(0)
        red = torch.zeros((1,), dtype=torch.float64, device=dev)

        def collect(t_, j):
            _lib.check(lib.ctcb_pipe_wait(ph, t_, None))
            if world > 1:                                   # the step's loss sum over all ranks, back on the host
                red.copy_(sum_bufs[j], non_blocking=True)
                dist.all_reduce(red)
                return float(red.item())
            return float(loss_np[j].sum())

        def pipe_run(k, record=False):
            acc, pending = 0.0, []
            for i in range(k):
                if world > 1:
                    sum_bufs[i % npb].zero_()
                _lib.check(lib.ctcb_pipe_submit(ph, ctypes.byref(pprobs[i % npb]), ctypes.byref(tk)))
                if record:
                    _lib.check(lib.ctcb_pipe_last_h2d_bytes(ph, ctypes.byref(hb), ctypes.byref(pulled)))
                    moved[i % npb] = hb.value
                pending.append((tk.value, i % npb))
                if len(pending) >= depth:
                    acc += collect(*pending.pop(0))
            for t_, j in pending:
                acc += collect(t_, j)
            return acc

        pipe_run(max(2 * depth, npb), record=True)
        # at least 200 steps whatever --steps says (12 ms at cfg2): the loop is timed with its fill and its drain, a fixed cost of
        # about one and a half steps that 20 steps would show as 6 % (61.8 against 57.9 us per step); the object reports its `steps`
        pipe_steps = max(e2e_steps, min(args.steps, 1000), 200)
        barrier()
        t0 = time.perf_counter()
        acc = pipe_run(pipe_steps)
        pipe_ms = (time.perf_counter() - t0) * 1e3
        pipe_frames = sum(frames_global[i % npb] for i in range(pipe_steps))
        if world > 1:
            a = torch.tensor([pipe_ms], dtype=torch.float64, device=dev)
            dist.all_reduce(a, op=dist.ReduceOp.MAX)
            pipe_ms = a[0].item()
        h2d_rank = sum(moved[i % npb] for i in range(pipe_steps)) / pipe_steps
        e2e_pipe = {"value": pipe_frames / (pipe_ms * 1e-3), "unit": UNIT, "ms_per_step": pipe_ms / pipe_steps,
                    "h2d_bytes_per_step": h2d_rank * world, "d2h_bytes_per_step": (d2h + 8) * world, "steps": pipe_steps,
                    "in_flight": depth, "loss_checksum": acc,
                    "h2d_bytes_per_step_dense": hsets[0].h2d_bytes * world,
                    "host_layout": ("dense (B,T,V) arena" if args.dense_host else
                                    "packed arena: the valid frames of every utterance back to back + int64 row offsets "
                                    "(ctcb_problem_t.logits_row_offsets); the dense gradient is formed on the device"),
                    "api": "ctcb_pipe_submit / ctcb_pipe_wait (pinned HOST batches, one cudaMemcpyAsync of the batch's arena): "
                           "every step's inputs cross PCIe and its loss is read on the host inside the timed region; batch "
                           "i+1's transfer overlaps batch i's kernels (%d in flight); gradient left on the device; host wall "
                           "clock around the loop including the drain%s" %
                           (depth, "; every step's loss sum all-reduced over the %d ranks (NCCL); bytes are the sum over ranks" % world if world > 1 else "")}
        lib.ctcb_pipe_destroy(ph)
    except Exception as exc:  # noqa: BLE001
        e2e_pipe = {"error": str(exc)[:200]}

    # ---- roofline of the dominant kernel: per-kernel CUDA events inside the library -------
    kms = np.zeros((8,), np.float64)
    nrep = 20
    kbuf = (ctypes.c_float * 8)()
    nk = ctypes.c_int32(0)
    alg = 0.0
    with torch.cuda.stream(stream):
        for i in range(nrep + 3):
            s = sets[i % nset]
            call = ops._Call(s["pred"], s["label"], s["pl"], s["ll"], False, True, False)
            ws = ops._ws_cache[(dev.index, stream.cuda_stream, call.T, call.B, call.V, call.Lmax)]
            p = call.problem(s["loss"], s["grad"], head)
            _lib.check(lib.ctcb_loss_grad_timed(ctypes.byref(p), ws.data_ptr(), ws.numel(), stream.cuda_stream,
                                                kbuf, ctypes.byref(nk)))
            if i >= 3:
                kms += np.array(list(kbuf))
                alg += algorithmic_bytes(V, T, B, s["np"]["pred_lengths"], s["np"]["label_lengths"])
    kms = kms[:nk.value] / nrep
    alg /= nrep
    gname = _lib.last_grad_kernel() or "k_grad"            # k_grad, or k_grad2 from 64 utterances per GPU on
    knames = ["k_emit", "k_walk", gname] if nk.value == 3 else ["k_walk", gname]
    dom = int(np.argmax(kms))
    peak, peak_src = measured_peak()
    achieved = alg / (kms[dom] * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            with open(tp) as f:
                tj = json.load(f)
            tw = tj.get(name, {})
            traffic = tw.get("whole_step", tw.get(knames[dom].replace("k_grad2", "k_grad"))) if world == 1 else None
            traffic_src = tj.get("_source")
        except Exception:
            traffic = None
    roofline = {
        "bound": "hbm", "kernel": knames[dom], "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": alg,
        "kernel_ms": {k: float(v) for k, v in zip(knames, kms)},
        "step_achieved": alg / (ms_per_step * 1e-3) / 1e9,
        "step_frac": alg / (ms_per_step * 1e-3) / 1e9 / peak,
        "note": "per GPU: this rank's algorithmic bytes over the step time; fp32 logits/gradient in HBM, fp64 linear-domain "
                "lattice recursion; the V=46 path is bound by the recursion's dependent chain and by instruction issue, not by "
                "HBM (SURVEY.md 8d / DESIGN.md sections 5-6); kernel_ms are the kernels timed one after the other, in the step "
                "k_grad runs concurrently with k_walk while the batch's walkers fit the GPU at once",
    }

    # ---- other workloads, same run (N=1 only): context numbers, not the headline ----------
    others = []
    next_rows = None
    if world == 1 and not args.no_others:
        for oname in ("cfg1", "cfg2", "cfg3", "cfg4", "cfg5"):
            if oname == name:
                continue
            try:
                others.append(measure_other(torch, ops, dev, oname, peak))
            except Exception as exc:  # noqa: BLE001
                others.append({"workload": oname, "error": str(exc)[:200]})
        try:
            next_rows = {"proj_ctc_forward": measure_proj(torch, dev)}
        except Exception as exc:  # noqa: BLE001
            next_rows = {"proj_ctc_forward": {"error": str(exc)[:200]}}
        c5 = next((o for o in others if o.get("workload") == "cfg5" and "value" in o), None)
        if c5:
            sweep = {"workload": "cfg5: one B=1024 batch (the sharded sweep of BASELINE configs[4]), whole batch on this GPU",
                     "n_gpus": 1, "ms_per_step": c5["ms_per_step"], "value": c5["value"], "unit": UNIT}

    cpu_baseline = None
    if rank == 0 and world == 1:
        ts, fr, cores, _ = time_cpu_rotation(name, 1000, 2, budget_s=10.0)
        cms = 1e3 * sum(ts) / len(ts)
        cpu_baseline = {"value": sum(fr) / sum(ts), "unit": UNIT, "cores": cores, "kind": "port",
                        "ms_per_step": cms,
                        "sample": "%d full %s steps (B=%d) of oracle/ctc_ref.c fp32, OpenMP over the minibatch" % (len(ts), name, Bg)}
        cpu_baseline.update(extra_cpu_baselines(sets[0]["np"], name))

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak" if world == 1 else "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(name, world, args.steps, frames_all / args.steps),
            "impl_notes": {
                "utterances_per_sec": Bg / (ms_per_step * 1e-3),
                "l2": "inputs rotate over %d buffer sets (%.0f MB logits+grad per rank > 126 MB L2)" % (nset, nset * per_set / 1e6),
                "launch": "%d kernels per step (k_grad a programmatic dependent of k_walk when the walkers fit the GPU at once) "
                          "%s; eager_ms_per_step=%.4f (no exchange)%s" %
                          (launches_per_step, "replayed from a CUDA graph" if use_graph else
                           "launched eagerly (step i+1's recursion kernel is the programmatic dependent of step i's gradient kernel)",
                           eager_ms, "; un-timed calibration over 30 steps: graph %.4f / eager %.4f ms per step" %
                           (calib["graph_ms_per_step"], calib["eager_ms_per_step"]) if calib else ""),
                "walker": {"pairs_per_lane": walk_cfg[0], "warps": walk_cfg[1]},
                "start_gate": "host barrier, then one un-timed all-reduce on the timed stream right before the start event" if world > 1 else ("a %.0f us hold kernel ahead of the start event: the first steps are queued behind it when the clock starts" % args.start_gate_us if args.start_gate_us > 0 else "none (one rank)"),
                "collective": ("none" if not exchange else
                               "none on the data path; float64 loss-sum exchange of the previous step's sum inside each step's CUDA graph: " +
                               ("ctcb_mailbox_exchange_with_next: a one-warp kernel stores the partial sums into every rank's mailbox over "
                                "NVLink peer memory and picks up the sums of %d steps before (no collective kernel, no rendezvous); it is the "
                                "programmatic dependent of the step's gradient kernel" % args.peer_lag
                                if collective == "peer" else "NCCL all-reduce (torch.distributed) on a side branch of the graph"))},
            "clocks": clocks,
            "e2e": (e2e_pipe if e2e_pipe and "value" in e2e_pipe else
                    e2e_cabi if e2e_cabi and "value" in e2e_cabi else e2e_plugin if e2e_plugin else e2e_pipe),
            "gpu_launches": (launches_per_step + (1 if (peer is not None and exchange) else 0)) * args.steps,
            "roofline": roofline,
        }
        if e2e_cabi:
            line["e2e_sync"] = e2e_cabi
        if e2e_plugin:
            line["e2e_plugin"] = e2e_plugin
        if sweep:
            line["sweep"] = sweep
        if cpu_baseline:
            line["cpu_baseline"] = cpu_baseline
        if others:
            line["other_workloads"] = others
        if next_rows:
            line["next_rows"] = next_rows
        print(json.dumps(line), flush=True)
    if world > 1:
        # The captured graphs hold NCCL work: tearing the communicator down under them can block, and a
        # rank that lingers would stall the launcher.  Everything is measured and printed; leave together.
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def measure_other(torch, ops, dev, oname, peak, steps=20, warmup=3):
    B, T, V, L = CONFIGS[oname]
    per_set = 2 * 4 * B * T * V
    nset = max(2, min(8, (2 * L2_BYTES + per_set - 1) // per_set + 1))
    sets = []
    for i in range(nset):
        d = make_batch(B, T, V, L, seed=i, full_lengths=(oname == "cfg5"))
        sets.append((torch.tensor(d["pred"], device=dev), torch.tensor(d["label"], device=dev),
                     torch.tensor(d["pred_lengths"], device=dev), torch.tensor(d["label_lengths"], device=dev),
                     torch.empty((B,), device=dev), torch.empty((B, T, V), device=dev),
                     float(d["pred_lengths"].sum()), algorithmic_bytes(V, T, B, d["pred_lengths"], d["label_lengths"])))
    head = torch.full((B,), 1.0 / B, device=dev)

    def step(s):
        ops.ctc_loss_and_grad(s[0], s[1], s[2], s[3], head_grad=head, out_loss=s[4], out_grad=s[5], handoff="pointer")
    for i in range(warmup):
        step(sets[i % nset])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(int(300e-6 * 1.9e9))      # the same hold kernel as ahead of the headline's start event: steps queued when the clock starts
    e0.record()
    frames = alg = 0.0
    for i in range(steps):
        s = sets[i % nset]
        step(s)
        frames += s[6]; alg += s[7]
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    ops._ws_cache.clear()
    del sets
    torch.cuda.empty_cache()
    return {"workload": oname, "B": B, "T": T, "V": V, "Lmax": L, "ms_per_step": ms / steps,
            "value": frames / (ms * 1e-3), "unit": UNIT, "step_achieved_gbs": alg / (ms * 1e-3) / 1e9,
            "step_frac": alg / (ms * 1e-3) / 1e9 / peak, "launch": "eager"}


def measure_proj(torch, dev, B=64, T=500, V=2000, L=150, H=512, steps=20, warmup=3):
    """SURVEY 8f rank 1 (context, not the headline): the output projection fused with the loss's forward
    (ctcb_proj_forward: tcgen05 tf32 GEMM whose epilogue feeds the lattice recursion, logits never stored) against the pair
    it replaces -- a library tf32 GEMM that writes the logits + ctcb_forward that reads them -- at BASELINE configs[2]'s
    shape with H hidden units.  Device-resident inputs, two buffer sets, CUDA events."""
    from gluon_e2e_asr_b200 import proj_ctc_loss
    from gluon_e2e_asr_b200.ops import ctc_loss
    sets = []
    for i in range(2):
        d = make_batch(B, T, V, L, seed=i)
        g = torch.Generator(device="cpu").manual_seed(i)
        sets.append((torch.randn((B, T, H), generator=g).to(dev), (torch.randn((V, H), generator=g) / H ** 0.5).to(dev),
                     torch.zeros((V,), device=dev), torch.tensor(d["label"], device=dev), torch.tensor(d["pred_lengths"], device=dev),
                     torch.tensor(d["label_lengths"], device=dev), float(d["pred_lengths"].sum())))
    old_tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True

    def fused(s):
        with torch.no_grad():
            return proj_ctc_loss(s[0], s[1], s[2], s[3], s[4], s[5])

    def unfused(s):
        with torch.no_grad():
            logits = torch.addmm(s[2], s[0].view(-1, H), s[1].t()).view(B, T, V)
            return ctc_loss(logits.transpose(0, 1), s[3], s[4], s[5], True, True)

    def gemm(s):
        return torch.addmm(s[2], s[0].view(-1, H), s[1].t())

    out = {"shape": {"B": B, "T": T, "V": V, "Lmax": L, "H": H}, "dtype": "tf32 product, fp32 accumulate, fp64 recursion"}
    try:
        for key, fn in (("fused_forward_us", fused), ("unfused_forward_us", unfused), ("library_gemm_us", gemm)):
            for i in range(warmup):
                fn(sets[i % 2])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                fn(sets[i % 2])
            e1.record()
            torch.cuda.synchronize()
            out[key] = e0.elapsed_time(e1) / steps * 1e3
        frames = 0.5 * (sets[0][6] + sets[1][6])
        out["valid_frames_per_step"] = frames
        out["fused_forward_frames_per_s"] = frames / out["fused_forward_us"] * 1e6
        out["max_rel_loss_difference"] = float(((fused(sets[0]) - unfused(sets[0])).abs() / unfused(sets[0]).abs().clamp_min(1)).max())
        out["projection_flops"] = 2.0 * B * T * H * V
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old_tf32
    del sets
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(CONFIGS),
                    help="default: cfg2 on one GPU (BASELINE configs[1]); cfg5 split by utterance on N > 1 (configs[4])")
    ap.add_argument("--pipe-depth", type=int, default=3, help="batches in flight in the prefetching host entry (e2e)")
    ap.add_argument("--start-gate-us", type=float, default=300.0,
                    help="one rank: length of the hold kernel ahead of the start event (0 = none)")
    ap.add_argument("--no-others", action="store_true", help="skip the context measurements of the other configs")
    ap.add_argument("--dense-host", action="store_true", help="e2e: dense (B,T,V) host batches instead of the packed arena")
    ap.add_argument("--collective", default="peer", choices=["peer", "nccl"],
                    help="N>1: loss-sum exchange through the library's peer mailbox (default) or torch.distributed's NCCL all-reduce")
    ap.add_argument("--peer-lag", type=int, default=4, help="slack between the ranks of the peer mailbox exchange, in steps")
    ap.add_argument("--no-allreduce", action="store_true", help="experiment: no loss-sum collective at all (N>1)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's losses and gradient to DIR as .npy files (one rank)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.dump_outputs and world > 1:
        ap.error("--dump-outputs writes the outputs of one process: run it with WORLD_SIZE=1")
    run_cuda(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
