"""Device-resident timings of CTC forced alignment, gtnb_ctc_align against the lattice route on the same inputs
(CUDA events, L2 flushed before every timed call).  The lattice route is what the project offered before:
gtnb_compose_linear of the CTC graphs (arcSort order, exact ties) + gtnb_viterbi_path, and + gtnb_forward
(tropical) for the scores that gtnb_ctc_align also returns.  Configs: the forced-alignment inputs of
scripts/bench_configs.py (B=64 T=2000 C=128 U=200) and the CTC benchmark's shape (B=256 T=1000 C=64 U=100).
Prints one JSON line per (config, route); the first line names the GPU, its power limit and max SM clock.
Before timing, the two routes' labels and scores are compared with == on the timed inputs.

    python scripts/bench_align.py [--iters N]
"""
import argparse
import ctypes as Ct
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gtn_b200 import capi  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from tests import util  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as ex:  # the timings stand without it
        return {"gpu": "unknown (%s)" % ex}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    args = ap.parse_args()
    L = capi.lib()
    ctx = capi.Ctx(0)
    print(json.dumps(gpu_info()), flush=True)

    def timeit(fn, n, warm=2):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(n):
            ctx.flush_l2()
            ctx.timer_start()
            fn()
            ts.append(ctx.timer_stop())
        return float(np.median(ts)), float(np.min(ts))

    for B, T, C, U, seed in ((64, 2000, 128, 200, 777), (256, 1000, 64, 100, 1234)):
        e, tg = util.bench_inputs(B, T, C, U, seed=seed)
        e_dev = ctx.to_device(e)
        lens = np.full(B, U, np.int32)
        cat = np.ascontiguousarray(np.concatenate(tg), np.int32)
        lab_dev = ctx.alloc(4 * B * T)
        st_dev = ctx.alloc(4 * B * T)
        scores = np.zeros(B, np.float32)

        def align():
            ctx._check(L.gtnb_ctc_align(ctx.h, B, T, C, e_dev.ptr, 1, None, cat.ctypes.data_as(capi._i32p),
                                        lens.ctypes.data_as(capi._i32p), 0, 1, lab_dev.ptr, st_dev.ptr, 1,
                                        scores.ctypes.data_as(capi._f32p)))

        views = [util.view_of(po.Graph.ctc(t, 0, True)) for t in tg]
        lat_out = {}

        def lattice(with_scores=True):
            lat = ctx.compose_linear(views, [T] * B, C, e_dev, T * C)
            lat_out["path"] = lat.viterbi_path(T)
            if with_scores:
                lat_out["scores"] = lat.forward(tropical=True)
            lat.free()

        align()
        lattice()
        labels = lab_dev.download((B, T), np.int32)
        same = bool(np.array_equal(labels, lat_out["path"]["ilabels"]) and np.array_equal(scores, lat_out["scores"]))
        cfg = {"B": B, "T": T, "C": C, "U": U, "outputs_equal": same}
        for name, fn, n in (("gtnb_ctc_align", align, args.iters),
                            ("lattice_path", lambda: lattice(False), max(3, args.iters // 3)),
                            ("lattice_path_and_score", lattice, max(3, args.iters // 3))):
            med, mn = timeit(fn, n)
            print(json.dumps(dict(cfg, route=name, ms_median=med, ms_min=mn, utt_per_s=B / (med * 1e-3),
                                  iters=n)), flush=True)
        for buf in (e_dev, lab_dev, st_dev):
            buf.free()
    ctx.close()


if __name__ == "__main__":
    main()
