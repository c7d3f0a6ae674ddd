#!/usr/bin/env python
"""bench.py -- CTC loss+gradient throughput, the metric of BASELINE.json.

  python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K --warmup W

One "step" = one pass of the hot path (benchmarks/ctc.cpp:150-165: parallelMap(fwd) +
parallelMap(bwd)) over one synthetic minibatch of B=256 utterances, T=1000, C=64, U=100 per
GPU (BASELINE.json configs[1]; weak scaling, so N GPUs = configs[4]'s 256/GPU).

  value   utterances/s with the emissions already resident in HBM (device pointers in,
          device gradients out, B losses read back)
  e2e     the same call with HOST buffers (pinned): H2D of the emissions and D2H of the
          gradients + losses inside the timed region
  roofline  the dominant kernel's algorithmic bytes / its CUDA-event time (DESIGN.md)
  cpu_baseline  the reference itself (oracle/_ref, parallelMap on all host threads) on a
          bounded sample of the same workload

Every timed region runs exactly --steps steps after --warmup untimed ones.  --dump-outputs DIR writes what
the device leg returned in its last timed step (see dump_outputs), so that two builds can be compared output
for output: the inputs are seeded, identical from run to run for the same arguments.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_DEF, C_DEF, U_DEF, B_DEF = 1000, 64, 100, 256


def make_inputs(first, count, T, C, U):
    e = np.empty((count, T, C), np.float32)
    tg = []
    for i in range(count):
        rng = np.random.default_rng(1234 + first + i)
        e[i] = rng.uniform(-5.0, 5.0, (T, C)).astype(np.float32)
        tg.append(rng.integers(1, C, U).astype(np.int32))
    return e, tg


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(path, outputs):
    """outputs: {name: array whose first axis is the utterance}, written as path/<name>.npy in float32 or
    float64 (integer outputs as float64, which holds them exactly).  When they exceed DUMP_BYTES together,
    every array keeps the same utterances: a sorted sample drawn with a fixed seed, as many as fit."""
    os.makedirs(path, exist_ok=True)
    outputs = {k: (v.astype(np.float64) if v.dtype.kind in "iu" else v) for k, v in outputs.items()}
    B = len(next(iter(outputs.values())))
    per_utt = sum(v.nbytes for v in outputs.values()) // B
    keep = np.arange(B)
    if per_utt * B > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(B, DUMP_BYTES // per_utt, replace=False))
    for k, v in outputs.items():
        np.save(os.path.join(path, k + ".npy"), np.ascontiguousarray(v[keep]))


def ctc_view(capi, target, blank=0):
    """The CTC target graph of benchmarks/ctc.cpp:40-58 as a C-ABI graph view (host arrays): 2U+1
    nodes, per node a self loop, the step arc and -- between different labels -- the skip arc."""
    U = len(target)
    L = 2 * U + 1
    flags = np.zeros(L, np.uint8)
    flags[0] |= 1
    flags[L - 1] |= 2
    if L > 1:
        flags[L - 2] |= 2
    src, dst, lab = [], [], []
    for l in range(L):
        label = int(target[(l - 1) // 2]) if l % 2 else blank
        src.append(l), dst.append(l), lab.append(label)
        if l > 0:
            src.append(l - 1), dst.append(l), lab.append(label)
        if l % 2 and l > 1 and label != int(target[(l - 3) // 2]):
            src.append(l - 2), dst.append(l), lab.append(label)
    src, dst, lab = (np.asarray(a, np.int32) for a in (src, dst, lab))
    A = len(src)

    def lists(key):  # arcs grouped by node, arc ids ascending: CSR pointers + arc list
        order = np.argsort(key, kind="stable").astype(np.int32)
        ptr = np.zeros(L + 1, np.int32)
        np.add.at(ptr, key + 1, 1)
        return np.cumsum(ptr).astype(np.int32), order

    in_ptr, in_arcs = lists(dst)
    out_ptr, out_arcs = lists(src)
    return capi.make_view(flags, src, dst, lab, lab, np.zeros(A, np.float32), in_ptr, in_arcs, out_ptr,
                          out_arcs, np.array([0], np.int32), np.nonzero(flags & 2)[0].astype(np.int32))


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md), through NVML
    (the counters nvidia-smi prints).  An NVML query stalls kernel submission for milliseconds
    (measured: a 50 ms polling thread turned 2.5 ms steps into a 4.5 ms mean), so samples are
    taken synchronously BETWEEN two event-bracketed steps -- the GPU has been under load for
    the whole region, and no step's CUDA-event bracket contains a query."""

    def __init__(self, index):
        self.index = index
        self.sm, self.reasons = [], set()
        self.mx = None
        self.h = None
        self.nv = None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            self.h = nv.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def sample(self):
        nv = self.nv
        if nv is None:
            return self._smi()
        try:
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for bit, nm in ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"),
                            (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap")):
                if r & bit:
                    self.reasons.add(nm)
        except Exception:
            pass

    def _smi(self):
        try:
            out = subprocess.run(
                ["nvidia-smi", "-i", str(self.index),
                 "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits"],
                capture_output=True, text=True, timeout=10).stdout.strip().split(",")
            self.sm.append(float(out[0]))
            self.mx = float(out[1])
            for k, nm in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
                if out[2 + k].strip().lower().startswith("active"):
                    self.reasons.add(nm)
        except Exception:
            pass

    def result(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples"], "samples": 0}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.mx, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "source": "nvml" if self.nv else "nvidia-smi",
                "when": "between event-bracketed steps of the timed region"}


def bind_to_gpu_numa_node(index):
    """One process per GPU: run this rank (and first-touch its pinned buffers) on the CPUs of the NUMA node the
    GPU hangs off.  torchrun does not bind ranks, and round 1's e2e scaling collapsed at N >= 4 because ranks
    of GPUs 4-7 were copying through the other socket.  Returns a description for the JSON line."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(index)
        bus = nv.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dev = "/sys/bus/pci/devices/" + bus.lower()[-12:]
        node = int(open(dev + "/numa_node").read())
        cpus = set()
        for part in open(dev + "/local_cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        use = (cpus & allowed) or allowed
        os.sched_setaffinity(0, use)
        return {"gpu": index, "numa_node": node, "cpus": len(use)}
    except Exception as ex:  # no sysfs entry (a VM), no NVML: run unbound
        return {"gpu": index, "numa_node": None, "error": str(ex)[:80]}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def workload_config(B, T, C, U, world):
    """The `config` object, identical for both arms (`--impl ours` / `--impl reference`)."""
    return {"workload": "CTC loss+grad B=%d/GPU T=%d C=%d U=%d (BASELINE.json configs[1]; x N GPUs = configs[4])"
                        % (B, T, C, U),
            "l2": "flushed between timed iterations (256 MB memset); inputs 65.5 MB < 126 MB L2",
            "parallelism": "dp%d" % world}


def cpu_reference(sample, T, C, U, repeats=1, keep=None):
    """The real reference (oracle/_ref) on `sample` utterances, all host threads.  keep (a dict):
    receives the reference's losses / gradients for the in-run parity block."""
    from oracle import pyoracle as po
    if not po.have_ref():
        po.build(ref=False)
        # the C restatement, single thread (kind "port")
        e, tg = make_inputs(0, min(sample, 8), T, C, U)
        t0 = time.perf_counter()
        for b in range(e.shape[0]):
            po.ctc_loss(e[b], tg[b], 0, True)
        dt = time.perf_counter() - t0
        return {"value": e.shape[0] / dt, "unit": "utt/s", "cores": 1, "kind": "port",
                "sample": "%d utterances T=%d C=%d U=%d, oracle/gtn_oracle.c" % (e.shape[0], T, C, U)}
    cores = po.libref().ref_hardware_threads()
    e, tg = make_inputs(0, sample, T, C, U)
    po.ref_ctc_batch(e[:min(sample, 2 * max(cores, 1))], tg[:min(sample, 2 * max(cores, 1))])  # warm the pool
    best = None
    for _ in range(repeats):
        lr, gr, sec = po.ref_ctc_batch(e, tg)
        best = sec if best is None else min(best, sec)
    if keep is not None:
        keep.update(losses=lr, grads=gr, e=e, tg=tg)
    return {"value": sample / best, "unit": "utt/s", "cores": min(cores, sample), "kind": "reference",
            "sample": "%d utterances T=%d C=%d U=%d via parallelMap on %d threads (benchmarks/ctc.cpp:150-165)"
                      % (sample, T, C, U, min(cores, sample)), "seconds": best}


def api_path_leg(e, tg, T, C, steps):
    """The drop-in path a user gets by swapping the import: the reference's Python surface (gtn_b200.gtn), one
    Graph per utterance, the LIST forms of intersect / forward_score / subtract / backward (bindings/python/
    gtn/_functions.cpp:69-135), emissions handed over as device pointers of a torch CUDA tensor
    (docs/source/pytorch.rst's set_weights(data_ptr)), gradients read back per utterance with
    weights_to_numpy() exactly as bindings/python/examples/pytorch_loss.py:83-102 does.  Target graphs are
    built once outside the timed region (Python-loop graph construction is interpreter time, not the path).
    Wall clock with a device synchronise on both sides (the gtn layer runs on its own streams)."""
    import torch
    import gtn_b200.gtn as gtn
    B = e.shape[0]
    x = torch.tensor(e, device="cuda")
    ctcs = []
    for t in tg:
        L = 2 * len(t) + 1
        g = gtn.Graph(False)
        for l in range(L):
            g.add_node(l == 0, l == L - 1 or l == L - 2)
            label = int(t[(l - 1) // 2]) if l % 2 else 0
            g.add_arc(l, l, label)
            if l > 0:
                g.add_arc(l - 1, l, label)
            if l % 2 and l > 1 and label != int(t[(l - 3) // 2]):
                g.add_arc(l - 2, l, label)
        g.arc_sort()
        ctcs.append(g)

    def step():
        ems = []
        for b in range(B):
            em = gtn.linear_graph(T, C)
            em.set_weights(x[b].data_ptr())
            ems.append(em)
        losses = gtn.subtract(gtn.forward_score(ems), gtn.forward_score(gtn.intersect(ctcs, ems)))
        gtn.backward(losses)
        grads = [em.grad().weights_to_numpy() for em in ems]
        return np.array([l.item() for l in losses], np.float32), grads

    step()
    l0 = gtn.device_launch_count()
    ts = []
    for _ in range(steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        losses, grads = step()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    launches = (gtn.device_launch_count() - l0) / steps
    ms = 1e3 * float(np.median(ts))
    return {"ms_per_step": ms, "utt_per_s": B / (ms * 1e-3), "steps": steps, "kernel_launches_per_step": launches,
            "what": "gtn_b200.gtn list overloads, B=%d Graphs, device-pointer emissions in, per-utterance host "
                    "gradients out (weights_to_numpy), target graphs prebuilt" % B,
            "clock": "wall, median"}, losses, grads


def parity_block(ctx, keep, losses_gpu, g_dev, T, C):
    """SURVEY.md 8(d) "parity check in the same run": the reference ran on the first n utterances of the
    very batch that was timed (same seeds); compare the losses and gradients of the LAST TIMED STEP of the
    device leg with it and -- on a few of them -- with the float64 referee (oracle/f64.py)."""
    from oracle import f64
    lr, gr = keep["losses"], keep["grads"]
    n = len(lr)
    go = g_dev.download((n, T, C))
    lo = losses_gpu[:n]
    rel = np.abs(lo - lr) / np.maximum(np.abs(lr), 1e-30)
    n64 = min(n, 16)
    ref_err = my_err = 0.0
    for b in range(n64):
        _, g64 = f64.ctc_f64(keep["e"][b], keep["tg"][b])
        ref_err = max(ref_err, float(np.abs(gr[b] - g64).max()))
        my_err = max(my_err, float(np.abs(go[b] - g64).max()))
    return {"n": int(n), "against": "oracle/_ref (the unmodified reference) on utterances 0..n-1 of the timed batch",
            "max_rel_loss": float(rel.max()), "max_abs_grad": float(np.abs(go - gr).max()),
            "n_f64": int(n64), "max_abs_grad_vs_f64": my_err, "ref_max_abs_grad_vs_f64": ref_err,
            "ok": bool(rel.max() <= 1e-4 and my_err <= 2.0 * ref_err + 1e-5),
            "bar": "loss 1e-4 relative; gradient at least as close to the float64 lattice evaluation as the "
                   "reference's own fp32 gradient is (x2) -- DESIGN.md Tolerances"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    T, C, U = args.T, args.C, args.U
    # same config as our arm: one step = the whole B-utterance minibatch through
    # parallelMap(fwd) + parallelMap(bwd) (benchmarks/ctc.cpp:150-165), ~1-7 s per step on the host
    sample = args.batch
    from oracle import pyoracle as po
    e, tg = make_inputs(0, sample, T, C, U)
    kind = "reference" if po.have_ref() else "port"
    if kind == "reference":
        cores = min(po.libref().ref_hardware_threads(), sample)
        step = lambda: po.ref_ctc_batch(e, tg)[2]
    else:
        cores = 1

        def step():
            t0 = time.perf_counter()
            for b in range(sample):
                po.ctc_loss(e[b], tg[b], 0, True)
            return time.perf_counter() - t0
    for _ in range(args.warmup):
        step()
    secs = [step() for _ in range(args.steps)]
    ms = 1e3 * float(np.mean(secs))
    val = sample / (ms / 1e3)
    print(json.dumps({
        "impl": "reference", "metric": "ctc_fwd_bwd_utterances_per_s", "value": val, "unit": "utt/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(sample, T, C, U, world),
        "ms_per_step_median": 1e3 * float(np.median(secs)), "ms_per_step_all": [1e3 * x for x in secs],
        "cpu_baseline": {"value": val, "unit": "utt/s", "cores": cores, "kind": kind,
                         "sample": "the full %d-utterance minibatch per step, %d steps" % (sample, args.steps)},
        "e2e": {"value": val, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------------------------
# the other BASELINE.json configurations: ASG (configs[2]) and dense Viterbi (configs[3])
# ---------------------------------------------------------------------------------------------------------

def run_other_workload(args, rank, local, world):
    """One JSON line for --workload asg | viterbi, same contract as the headline: `value` device resident,
    `e2e` with pinned host buffers, `roofline` for the dominant kernel, `cpu_baseline` = the reference
    (oracle/_ref) on a bounded sample, in-run `parity` against it.  Weak scaling (B per GPU)."""
    asg = args.workload == "asg"
    B = args.batch if args.batch != B_DEF else (128 if asg else 512)
    T = args.T if args.T != T_DEF else (500 if asg else 2000)
    C = args.C if args.C != C_DEF else (64 if asg else 128)
    U = args.U if args.U != U_DEF else 50
    name = ("ASG loss+grad B=%d/GPU T=%d C=%d U=%d (BASELINE.json configs[2])" % (B, T, C, U)) if asg else \
           ("dense Viterbi score+path B=%d/GPU T=%d C=%d (BASELINE.json configs[3])" % (B, T, C))
    metric = "asg_fwd_bwd_utterances_per_s" if asg else "viterbi_decode_utterances_per_s"
    rngw = np.random.default_rng(7)
    tw = rngw.uniform(-5, 5, C + C * C).astype(np.float32)

    def inputs(first, count):
        e = np.empty((count, T, C), np.float32)
        tg = []
        for i in range(count):
            rng = np.random.default_rng(4321 + first + i)
            e[i] = rng.uniform(-5.0, 5.0, (T, C)).astype(np.float32)
            tg.append(rng.integers(0, C, U).astype(np.int32))
        return e, tg

    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import pyoracle as po
        n = min(args.cpu_sample, 16 if asg else 8)
        e, tg = inputs(0, n)
        step = (lambda: po.ref_asg_batch(e, tw, tg)[3]) if asg else (lambda: po.ref_viterbi_dense_batch(e, tw)[2])
        for _ in range(args.warmup):
            step()
        secs = [step() for _ in range(args.steps)]
        val = n / float(np.mean(secs))
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": val, "unit": "utt/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(secs)),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": name, "parallelism": "dp%d" % world},
            "cpu_baseline": {"value": val, "unit": "utt/s", "cores": min(po.libref().ref_hardware_threads(), n),
                             "kind": "reference", "sample": "%d utterances per step (BASELINE.md: the CPU needs seconds "
                             "and gigabytes per utterance here)" % n},
            "e2e": {"value": val, "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import ctypes as Ct
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from gtn_b200 import capi
    L = capi.lib()
    ctx = capi.Ctx(local)
    i32p, f32p = capi._i32p, capi._f32p
    e, tg = inputs(rank * B, B)
    lens = np.full(B, U, np.int32)
    cat = np.ascontiguousarray(np.concatenate(tg), np.int32)
    e_dev = ctx.to_device(e)
    hp_e = Ct.c_void_p()
    ctx._check(L.gtnb_host_alloc(ctx.h, e.nbytes, Ct.byref(hp_e)))
    Ct.memmove(hp_e.value, e.ctypes.data, e.nbytes)
    losses = np.zeros(B, np.float32)
    if asg:
        g_dev = ctx.alloc(e.nbytes)
        hp_g = Ct.c_void_p()
        ctx._check(L.gtnb_host_alloc(ctx.h, e.nbytes, Ct.byref(hp_g)))
        tgrad = np.zeros(C + C * C, np.float32)

        def call(ep, eon, gp, gon):
            ctx._check(L.gtnb_asg_loss(ctx.h, B, T, C, ep, eon, tw.ctypes.data_as(f32p), cat.ctypes.data_as(i32p),
                                       lens.ctypes.data_as(i32p), losses.ctypes.data_as(f32p), gp, gon,
                                       tgrad.ctypes.data_as(f32p)))
        step_dev = lambda: call(e_dev.ptr, 1, g_dev.ptr, 1)
        step_e2e = lambda: call(hp_e.value, 0, hp_g.value, 0)
        h2d, d2h = e.nbytes + tw.nbytes + cat.nbytes, e.nbytes + losses.nbytes + tgrad.nbytes
        # SURVEY.md 8(d) B_io on the two factored lattices: emissions in, gradients out, per-frame node scores
        # (C for the denominator trellis, U for the forced-alignment chain) written once and read once
        alg = B * (4 * T * C + 4 * T * C + 2 * 4 * T * (C + U))
    else:
        paths = np.zeros((B, T), np.int32)
        scores = np.zeros(B, np.float32)

        def call(ep, eon):
            ctx._check(L.gtnb_viterbi_dense(ctx.h, B, T, C, ep, eon, None, tw.ctypes.data_as(f32p),
                                            paths.ctypes.data_as(i32p), scores.ctypes.data_as(f32p)))
        step_dev = lambda: call(e_dev.ptr, 1)
        step_e2e = lambda: call(hp_e.value, 0)
        h2d, d2h = e.nbytes + tw.nbytes, paths.nbytes + scores.nbytes
        # emissions in, one back-pointer byte per (frame, state) written and read by the traceback, paths out
        alg = B * (4 * T * C + 2 * T * C + 4 * T)

    for _ in range(args.warmup):
        step_dev()
    sampler = ClockSampler(local)
    every = max(1, args.steps // 8)

    def region(step, profile):
        if profile:
            ctx.profile(True)
            ctx.profile_read()
        l0 = ctx.launches
        barrier()
        ts, pr = [], {}
        for i in range(args.steps):
            ctx.flush_l2()
            ctx.timer_start()
            step()
            ts.append(ctx.timer_stop())
            if profile:
                for k, (cnt, ms_) in ctx.profile_read().items():
                    c0, m0 = pr.get(k, (0, 0.0))
                    pr[k] = (c0 + cnt, m0 + ms_)
            if i % every == every // 2:
                sampler.sample()
        barrier()
        if profile:
            ctx.profile(False)
        return ts, pr, ctx.launches - l0

    ts, pr, launches = region(step_dev, True)
    gpu_losses = losses.copy() if asg else scores.copy()
    gpu_paths = None if asg else paths.copy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"losses": gpu_losses, "grads": g_dev.download((B, T, C))} if asg else
                     {"scores": gpu_losses, "paths": gpu_paths})
        if asg:
            np.save(os.path.join(args.dump_outputs, "transition_grads.npy"), tgrad)
    for _ in range(2):
        step_e2e()
    te, _, _ = region(step_e2e, False)
    ms, ems = float(np.mean(ts)), float(np.mean(te))
    if world > 1:
        t = torch.tensor([ms, ems], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ems = float(t[0]), float(t[1])
    if rank == 0:
        peak, peak_src = load_peaks()
        kern = {k: v[1] / args.steps for k, v in pr.items() if k != "flush_l2"}
        dom = max(kern.items(), key=lambda kv: kv[1]) if kern else (None, 0.0)
        out = {
            "metric": metric, "value": world * B / (ms * 1e-3), "unit": "utt/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "ms_per_step_median": float(np.median(ts)),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": name, "l2": "flushed between timed iterations (256 MB memset)",
                       "parallelism": "dp%d" % world},
            "e2e": {"value": world * B / (ems * 1e-3), "unit": "utt/s", "ms_per_step": ems,
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches), "clocks": sampler.result(),
            # the factored lattices move almost nothing: the sweeps are bound by SFU / issue rate and per-frame
            # latency (SURVEY.md 8(d)); the HBM figure is reported against the WHOLE step for completeness
            "roofline": {"bound": "hbm", "kernel": "whole step (dominant kernel by time: %s, %.3f ms)" % dom,
                         "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes": alg,
                         "note": "factored lattice: issue / SFU and per-frame latency bound, not HBM (SURVEY.md 8(d))"},
            "kernels_ms_per_step": kern}
        if not args.no_cpu_baseline:
            from oracle import pyoracle as po
            if po.have_ref():
                n = min(args.cpu_sample, 16 if asg else 8)
                if asg:
                    lr, gr, tgr, sec = po.ref_asg_batch(e[:n], tw, tg[:n])
                    go = g_dev.download((n, T, C))
                    out["parity"] = {"n": n, "max_rel_loss": float((np.abs(gpu_losses[:n] - lr) / np.abs(lr)).max()),
                                     "max_abs_grad": float(np.abs(go - gr).max()),
                                     "against": "oracle/_ref on utterances 0..n-1 of the timed batch (the transition "
                                                "gradient sums over a different batch and is compared in tests/)"}
                else:
                    pr_, sr, sec = po.ref_viterbi_dense_batch(e[:n], tw)
                    out["parity"] = {"n": n, "paths_equal": bool(np.array_equal(gpu_paths[:n], pr_)),
                                     "scores_equal": bool(np.array_equal(gpu_losses[:n], sr)),
                                     "against": "oracle/_ref on utterances 0..n-1 of the timed batch, =="}
                out["cpu_baseline"] = {"value": n / sec, "unit": "utt/s", "kind": "reference", "seconds": sec,
                                       "cores": min(po.libref().ref_hardware_threads(), n),
                                       "sample": "%d utterances on %d threads (BASELINE.md section 3)" % (n, min(po.libref().ref_hardware_threads(), n))}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=None,
                    help="utterances per GPU (default %d); with --strong: of the whole job (default 2048 = configs[4])" % B_DEF)
    ap.add_argument("--T", type=int, default=T_DEF)
    ap.add_argument("--C", type=int, default=C_DEF)
    ap.add_argument("--U", type=int, default=U_DEF)
    ap.add_argument("--cpu-sample", type=int, default=64)
    ap.add_argument("--workload", default="ctc", choices=["ctc", "asg", "viterbi"],
                    help="ctc: BASELINE configs[1] (the headline, what the driver runs); asg: configs[2]; "
                         "viterbi: configs[3]")
    ap.add_argument("--strong", action="store_true",
                    help="ctc only: --batch is the WHOLE job (configs[4]: B=2048 fixed), split over the ranks")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-api-path", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of the device leg as DIR/<name>.npy (rank 0's; "
                         "at most 64 MB: above that, the same seeded sample of utterances of every output)")
    args = ap.parse_args()
    if args.batch is None:
        args.batch = 2048 if args.strong else B_DEF

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.workload != "ctc":
        run_other_workload(args, rank, local, world)
        return
    if args.strong:
        if args.batch % world:
            raise SystemExit("--strong: --batch must be a multiple of the number of ranks")
        args.total_batch = args.batch
        args.batch //= world
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"  # keeps NCCL's banner out of stdout: rank 0 prints ONE JSON line
    numa = bind_to_gpu_numa_node(local)  # before the first allocation: pinned buffers are first-touch
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from gtn_b200 import capi
    L = capi.lib()
    import ctypes as Ct
    ctx = capi.Ctx(local)
    B, T, C, U = args.batch, args.T, args.C, args.U
    e, tg = make_inputs(rank * B, B, T, C, U)
    lens = np.full(B, U, np.int32)
    cat = np.ascontiguousarray(np.concatenate(tg), np.int32)
    nbytes = e.nbytes
    e_dev = ctx.to_device(e)
    g_dev = ctx.alloc(nbytes)
    losses = np.zeros(B, np.float32)

    # pinned host buffers for the end-to-end leg
    hp_e, hp_g = Ct.c_void_p(), Ct.c_void_p()
    ctx._check(L.gtnb_host_alloc(ctx.h, nbytes, Ct.byref(hp_e)))
    ctx._check(L.gtnb_host_alloc(ctx.h, nbytes, Ct.byref(hp_g)))
    Ct.memmove(hp_e.value, e.ctypes.data, nbytes)

    i32p, f32p = capi._i32p, capi._f32p

    def step_dev():
        ctx._check(L.gtnb_ctc_loss(ctx.h, B, T, C, e_dev.ptr, 1, None, cat.ctypes.data_as(i32p),
                                   lens.ctypes.data_as(i32p), 0, losses.ctypes.data_as(f32p),
                                   g_dev.ptr, 1))

    def step_e2e():
        ctx._check(L.gtnb_ctc_loss(ctx.h, B, T, C, hp_e.value, 0, None, cat.ctypes.data_as(i32p),
                                   lens.ctypes.data_as(i32p), 0, losses.ctypes.data_as(f32p),
                                   hp_g.value, 0))

    # lattice sizes for the algorithmic byte counts (untimed): compose the same batch once through
    # the lattice API and read the node / arc counts back
    views = [ctc_view(capi, t, 0) for t in tg]
    lat = ctx.compose_linear(views, [T] * B, C, e_dev, T * C)
    nn, na = lat.sizes()
    lat.free()
    sumN, sumA = int(nn.sum()), int(na.sum())
    TC = T * C
    pitch = (2 * U + 1 + 3) // 4 * 4
    alg_bytes = {  # per launch, whole batch -- SURVEY.md section 8(d), DESIGN.md "Algorithmic bytes"
        "sd_forward": 8 * sumA + 12 * sumN,
        "sd_backward": 12 * sumA + 16 * sumN,
        # shortestDistanceGrad + compose gradFunc fused (criterion path): arc records, row_ptr,
        # saved scores in; emission gradients out (no arc gradients, no provenance in steady frames)
        "sd_backward_fused": 8 * sumA + 8 * sumN + 4 * TC * B,
        "compose_grad": 12 * sumA + 4 * sumN + 4 * TC * B,
        "compose_emit": 16 * sumA + 4 * sumN + 4 * TC * B,
        "linear_rows": 8 * TC * B,
        # implicit-lattice criterion kernels (k_implicit.cu): SURVEY.md 8(d) "B_io" -- emissions in,
        # dense per-frame node scores out (forward) / in (backward), emission gradients out
        # the bidirectional kernel (k_bidir.cu): the WHOLE criterion -- SURVEY.md 8(d) B_io = emissions in
        # (4TC), gradients out (4TC), per-frame node scores written once and read once (2 * 4 * T * S)
        "bidir_ctc": 4 * TC * B + 4 * TC * B + 2 * 4 * T * pitch * B,
        "implicit_forward": 4 * TC * B + 4 * (T + 1) * pitch * B,
        "implicit_backward": 4 * TC * B + 4 * (T + 1) * pitch * B + 4 * TC * B,
    }
    formulation = {"bidir_ctc": "B_io (lattice never materialised; SURVEY.md 8(d) secondary figure, whole criterion)",
                   "implicit_forward": "B_io (lattice never materialised)",
                   "implicit_backward": "B_io (lattice never materialised)"}
    b_csr = 32 * sumA + 28 * sumN + 12 * TC * B

    for _ in range(args.warmup):
        step_dev()
    ctx.synchronize()

    sampler = ClockSampler(local)
    every = max(1, args.steps // 8)

    def timed_region(step, profile):
        """EXACTLY args.steps steps, each bracketed by CUDA events on the launching stream (L2
        flushed before the bracket), barrier + synchronize on both sides of the region."""
        if profile:
            ctx.profile(True)
            ctx.profile_read()
        l0 = ctx.launches
        barrier()
        ts = []
        pr = {} if profile else None
        w0 = time.perf_counter()
        for i in range(args.steps):
            ctx.flush_l2()  # inputs (65.5 MB) are smaller than the 126 MB L2
            ctx.timer_start()
            step()
            ts.append(ctx.timer_stop())
            if profile:
                # between two brackets: read this step's per-kernel events and hand them back to the
                # pool, so that no step of the region pays for creating events
                for k, (cnt, ms_) in ctx.profile_read().items():
                    c0, m0 = pr.get(k, (0, 0.0))
                    pr[k] = (c0 + cnt, m0 + ms_)
            if i % every == every // 2:
                sampler.sample()
        barrier()
        w = time.perf_counter() - w0
        if profile:
            ctx.profile(False)
        return {"times": ts, "wall": w, "launches": ctx.launches - l0, "prof": pr}

    dev = timed_region(step_dev, True)
    times, wall, launches, prof = dev["times"], dev["wall"], dev["launches"], dev["prof"]
    losses_dev_leg = losses.copy()  # the last timed step's losses; its gradients are still in g_dev

    # end-to-end leg (host buffers)
    for _ in range(2):
        step_e2e()
    e2e = timed_region(step_e2e, False)
    e2e_times = e2e["times"]
    clocks = sampler.result()

    ms = float(np.mean(times))
    e2e_ms = float(np.mean(e2e_times))
    if os.environ.get("GTNB_BENCH_DUMP"):
        np.save(os.environ["GTNB_BENCH_DUMP"] + "_r%d.npy" % rank, np.array([times, e2e_times]))
    if world > 1:
        t = torch.tensor([ms, e2e_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0]), float(t[1])

    if rank == 0:
        peak, peak_src = load_peaks()
        # DRAM bytes per launch measured by `ncu --set full` (dram__bytes_read.sum +
        # dram__bytes_write.sum), committed with the ncu summary they come from
        traffic = {}
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp) and (B, T, C, U) == (B_DEF, T_DEF, C_DEF, U_DEF):
            traffic = json.load(open(tp)).get("bytes_per_launch", {})
        # dominant kernel by CUDA-event time
        dom = max(prof.items(), key=lambda kv: kv[1][1]) if prof else (None, (0, 0.0))
        name, (cnt, tot_ms) = dom
        roofline = None
        if name in alg_bytes and cnt:
            per_launch_ms = tot_ms / cnt
            ach = alg_bytes[name] / (per_launch_ms * 1e-3) / 1e9
            roofline = {"bound": "hbm", "kernel": name, "achieved": ach, "peak": peak, "unit": "GB/s",
                        "frac": ach / peak, "traffic": traffic.get(name), "peak_source": peak_src,
                        "kernel_ms": per_launch_ms, "algorithmic_bytes": alg_bytes[name],
                        "formulation": formulation.get(name, "B_csr (materialised lattice)"),
                        # the same step judged on the materialised-CSR byte count of SURVEY.md 8(d)
                        "step_csr_equiv_GBps": b_csr / (ms * 1e-3) / 1e9}
        kernels = {k: {"launches_per_step": v[0] / args.steps, "ms_per_step": v[1] / args.steps,
                       "GBps": (alg_bytes[k] / (v[1] / v[0] * 1e-3) / 1e9) if k in alg_bytes and v[0] else None}
                   for k, v in prof.items()}
        out = {
            "metric": "ctc_fwd_bwd_utterances_per_s", "value": world * B / (ms * 1e-3), "unit": "utt/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(B, T, C, U, world) if not args.strong else
            {"workload": "CTC loss+grad B=%d TOTAL (BASELINE.json configs[4]), %d per GPU, T=%d C=%d U=%d"
                         % (args.total_batch, B, T, C, U),
             "l2": "flushed between timed iterations (256 MB memset)", "parallelism": "dp%d" % world},
            "lattice": {"nodes": sumN, "arcs": sumA, "note": "per GPU, what compose would materialise"},
            "e2e": {"value": world * B / (e2e_ms * 1e-3), "unit": "utt/s", "ms_per_step": e2e_ms,
                    "ms_per_step_median": float(np.median(e2e_times)), "ms_per_step_min": float(np.min(e2e_times)),
                    "h2d_bytes_per_step": int(nbytes + cat.nbytes + lens.nbytes),
                    "d2h_bytes_per_step": int(nbytes + losses.nbytes)},
            "gpu_launches": int(launches),
            "numa": numa,
            "clocks": clocks,
            "ms_per_step_median": float(np.median(times)), "ms_per_step_min": float(np.min(times)),
            "roofline": roofline,
            "roofline_whole_step_csr": {"achieved": b_csr / (ms * 1e-3) / 1e9, "unit": "GB/s",
                                        "frac": b_csr / (ms * 1e-3) / 1e9 / peak, "bytes": b_csr},
            "kernels": kernels,
            "wall_s": wall,
        }
        if not args.no_cpu_baseline:
            keep = {}
            out["cpu_baseline"] = cpu_reference(args.cpu_sample, T, C, U, keep=keep)
            if keep:
                out["parity"] = parity_block(ctx, keep, losses_dev_leg, g_dev, T, C)
        if not args.no_api_path and world == 1:
            try:
                api, al, ag = api_path_leg(e, tg, T, C, args.steps)
                api["max_rel_loss_vs_fused"] = float((np.abs(al - losses_dev_leg) / np.abs(losses_dev_leg)).max())
                api["max_abs_grad_vs_fused"] = float(np.abs(np.stack(ag[:16]).reshape(16, T, C) - g_dev.download((16, T, C))).max())
                out["api_path"] = api
            except Exception as ex:  # the line must still print
                out["api_path"] = {"error": str(ex)[:200]}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"losses": losses_dev_leg, "grads": g_dev.download((B, T, C))})
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
