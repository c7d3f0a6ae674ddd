"""Helpers shared by the tests: graph builders, tolerances and the golden fixtures."""
import functools
import json
import os

import numpy as np

from gtn_b200 import capi

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GRAPH_KEYS = ("flags", "src", "dst", "ilabel", "olabel", "w")


@functools.lru_cache(maxsize=None)
def golden_host():
    """tests/golden/reference_host.json: the reference's outputs for the seeded host-side graph tests."""
    with open(os.path.join(GOLDEN, "reference_host.json")) as f:
        return json.load(f)


def golden_configs():
    """tests/golden/reference_configs.npz: the reference's outputs at the BASELINE.json configurations."""
    return np.load(os.path.join(GOLDEN, "reference_configs.npz"))


def graph_arrays(rec):
    """A graph stored in a golden fixture, [flags, src, dst, ilabel, olabel, w] -> dict of arrays."""
    return {k: np.array(v, np.float32 if k == "w" else (np.uint8 if k == "flags" else np.int32))
            for k, v in zip(GRAPH_KEYS, rec)}

# north_star tolerance: 1e-4 relative for scores and gradients; the small
# absolute term is the one the reference's own tests use (criterion_test.cpp:127)
RTOL = 1e-4
ATOL = 1e-5


def close(a, b, rtol=RTOL, atol=ATOL):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    both_nan = np.isnan(a) & np.isnan(b)
    same_inf = np.isinf(a) & np.isinf(b) & (np.sign(a) == np.sign(b))
    ok = np.abs(a - b) <= rtol * np.maximum(np.abs(a), np.abs(b)) + atol
    return bool(np.all(ok | both_nan | same_inf))


def ulp32(x):
    return float(np.spacing(np.float32(abs(x))))


def grad_close(a, b, score_mag):
    """Gradient parity with the conditioning of the fp32 recursion made explicit.

    Both the reference and the CUDA path evaluate exp(score[src] + w - max) on fp32
    node scores, so one ulp of the largest score bounds how well ANY two fp32
    evaluations can agree (measured: the reference itself is 1.9e-3 abs / 7.6e-2 rel
    off the float64 gradient at T=1000, C=64 -- DESIGN.md "Tolerances").  The bar is
    1e-4 relative plus an absolute term of 1e-5 (criterion_test.cpp:127) + 4 ulp(score).
    """
    return close(a, b, rtol=RTOL, atol=ATOL + 4.0 * ulp32(score_mag))


def view_of(og):
    """capi view of an oracle graph (oracle.pyoracle.Graph), keeping its arc-list order."""
    a = og.arrays()
    ip, ia, op, oa = og.adjacency()
    return capi.make_view(a["flags"], a["src"], a["dst"], a["ilabel"], a["olabel"], a["w"],
                          ip, ia, op, oa, a["start"], a["accept"])


def random_dag(rng, n_nodes, n_arcs, n_labels=3, int_weights=False):
    """Connected random DAG like benchmarks/time_utils.h:55-72 (makeRandomDAG)."""
    flags = np.zeros(n_nodes, np.uint8)
    flags[0] = 1
    flags[-1] |= 2
    src, dst = [], []
    for n in range(1, n_nodes):
        src.append(n - 1)
        dst.append(n)
    for _ in range(max(0, n_arcs - (n_nodes - 1))):
        s = int(rng.integers(0, n_nodes - 1))
        d = int(rng.integers(s + 1, n_nodes))
        src.append(s)
        dst.append(d)
    lab = rng.integers(0, n_labels, len(src)).astype(np.int32)
    if int_weights:
        w = rng.integers(-3, 4, len(src)).astype(np.float32)
    else:
        w = rng.uniform(-2, 2, len(src)).astype(np.float32)
    return flags, np.asarray(src, np.int32), np.asarray(dst, np.int32), lab, lab.copy(), w


def bench_inputs(B, T, C, U, seed=1234):
    """Synthetic CTC batch of SURVEY.md section 8(d): emissions U(-5,5), targets in [1, C-1]."""
    e = np.empty((B, T, C), np.float32)
    tg = []
    for b in range(B):
        rng = np.random.default_rng(seed + b)
        e[b] = rng.uniform(-5.0, 5.0, (T, C)).astype(np.float32)
        tg.append(rng.integers(1, C, U).astype(np.int32))
    return e, tg
