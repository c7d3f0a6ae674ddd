"""k_gcompose.cu (general device composition: epsilons, cycles, any sortedness) run on the CPU through the SIMT
emulator, against the reference (detail::compose, compose.cpp:377-522, its results on these seeded operands stored in
tests/golden/reference_host.json): identical node numbering, arc numbering, labels, weights and gradInfo -- not merely
isomorphic graphs."""
import ctypes as C

import numpy as np
import pytest

from tests import emu_build, util
from tests.test_host_api import golden, ours_arrays, ours_from, random_graph

i32p, f32p, u8p = C.POINTER(C.c_int32), C.POINTER(C.c_float), C.POINTER(C.c_uint8)


class EmuGraph(C.Structure):
    _fields_ = [("N", C.c_int32), ("A", C.c_int32), ("flags", u8p), ("src", i32p), ("dst", i32p), ("il", i32p),
                ("ol", i32p), ("w", f32p), ("in_ptr", i32p), ("in_arcs", i32p), ("out_ptr", i32p), ("out_arcs", i32p),
                ("start", i32p), ("n_start", C.c_int32), ("accept", i32p), ("n_accept", C.c_int32)]


@pytest.fixture(scope="module")
def gtn():
    import gtn_b200.gtn as g
    return g


@pytest.fixture(scope="module")
def emu():
    lib = C.CDLL(emu_build.build('gcompose', ['k_gcompose.cu', 'gtnb_gcompose.h']))
    lib.emu_gcompose.argtypes = [C.POINTER(EmuGraph), C.POINTER(EmuGraph), C.c_int, C.c_int, C.c_int, C.c_int, i32p, i32p, u8p,
                                 i32p, i32p, i32p, i32p, f32p, i32p, i32p]
    return lib


def pack(gtn, g):
    """EmuGraph of one of our Graphs: its arrays + g.in(n) / g.out(n) in the Graph's current order."""
    a = ours_arrays(g)
    lists = gtn.arc_lists(g)
    keep = [np.ascontiguousarray(a[k], t) for k, t in (("flags", np.uint8), ("src", np.int32), ("dst", np.int32),
                                                       ("ilabel", np.int32), ("olabel", np.int32), ("w", np.float32))]
    keep += [np.ascontiguousarray(lists[k], np.int32) for k in ("in_ptr", "in_arcs", "out_ptr", "out_arcs", "start", "accept")]
    ptr = lambda x, t: x.ctypes.data_as(t)
    eg = EmuGraph(len(keep[0]), len(keep[1]), ptr(keep[0], u8p), ptr(keep[1], i32p), ptr(keep[2], i32p), ptr(keep[3], i32p),
                  ptr(keep[4], i32p), ptr(keep[5], f32p), ptr(keep[6], i32p), ptr(keep[7], i32p), ptr(keep[8], i32p),
                  ptr(keep[9], i32p), ptr(keep[10], i32p), len(keep[10]), ptr(keep[11], i32p), len(keep[11]))
    return eg, keep


def kind_of(ga, gb, intersect):
    s1 = (ga.ilabel_sorted() or ga.olabel_sorted()) if intersect else ga.olabel_sorted()
    s2 = (gb.ilabel_sorted() or gb.olabel_sorted()) if intersect else gb.ilabel_sorted()
    return 3 if (s1 and s2) else (1 if s1 else (2 if s2 else 0))


def run(emu, gtn, ga, gb, intersect, cap=1 << 16, reach_ctas=1):
    ea, ka = pack(gtn, ga)
    eb, kb = pack(gtn, gb)
    nn, na = C.c_int32(0), C.c_int32(0)
    fl = np.zeros(cap, np.uint8)
    ints = [np.zeros(cap, np.int32) for _ in range(6)]
    w = np.zeros(cap, np.float32)
    rc = emu.emu_gcompose(C.byref(ea), C.byref(eb), kind_of(ga, gb, intersect), reach_ctas, cap, cap, C.byref(nn), C.byref(na),
                          fl.ctypes.data_as(u8p), ints[0].ctypes.data_as(i32p), ints[1].ctypes.data_as(i32p),
                          ints[2].ctypes.data_as(i32p), ints[3].ctypes.data_as(i32p), w.ctypes.data_as(f32p),
                          ints[4].ctypes.data_as(i32p), ints[5].ctypes.data_as(i32p))
    emu_build.check(rc)
    N, A = nn.value, na.value
    return dict(flags=fl[:N], src=ints[0][:A], dst=ints[1][:A], ilabel=ints[2][:A], olabel=ints[3][:A], w=w[:A],
                gi1=ints[4][:A], gi2=ints[5][:A])


def check_against(out, want, what):
    for k in ("flags", "src", "dst", "ilabel", "olabel", "w"):
        assert out[k].shape == want[k].shape, (what, k, out[k].shape, want[k].shape)
        assert np.array_equal(out[k], want[k]), (what, k, out[k], want[k])


def case(rng, seed, n_max, a_max, p_eps):
    a = random_graph(rng, int(rng.integers(1, n_max)), int(rng.integers(0, a_max)), n_labels=3, p_eps=p_eps)
    b = random_graph(rng, int(rng.integers(1, n_max)), int(rng.integers(0, a_max)), n_labels=3, p_eps=p_eps)
    intersect = seed % 3 == 0
    if intersect:  # acceptors
        a = (a[0], a[1], a[2], a[3], a[3].copy(), a[5])
        b = (b[0], b[1], b[2], b[3], b[3].copy(), b[5])
    return a, b, intersect


@pytest.mark.parametrize("seed", range(24))
def test_kernel_source_reproduces_the_reference_numbering(emu, gtn, seed):
    """Small arbitrary graphs, all three matchers (functions.cpp:225-251), epsilons on both sides."""
    rng = np.random.default_rng(700 + seed)
    a, b, intersect = case(rng, seed, 7, 14, 0.2)
    ma, mb = ours_from(gtn, a), ours_from(gtn, b)
    if seed & 1:
        ma.arc_sort(True)
    if seed & 2:
        mb.arc_sort(False)
    # every third case: the co-reachability search on 2 or 3 concurrent CTAs (gcompose_reach_kernel)
    out = run(emu, gtn, ma, mb, intersect, reach_ctas=(1, 1, 2, 1, 1, 3)[seed % 6])
    # the host construction of the gtn:: layer (pinned against the reference by tests/test_host_api.py)
    gtn.set_compose_device_policy(2)
    try:
        host = gtn.intersect(ma, mb) if intersect else gtn.compose(ma, mb)
    finally:
        gtn.set_compose_device_policy(0)
    check_against(out, ours_arrays(host), "vs the host construction")
    want = golden("compose", seed)
    check_against(out, util.graph_arrays(want["out"]), "vs the reference")
    # gradInfo (compose.cpp:445, 201-205): the scatter of random deltas equals the reference's backward
    assert (want["grads"] is not None) == bool(len(out["src"]))
    if len(out["src"]):
        d = rng.integers(-5, 6, len(out["src"])).astype(np.float32)
        for gi, wg, n in ((out["gi1"], want["grads"][0], len(a[1])), (out["gi2"], want["grads"][1], len(b[1]))):
            g = np.zeros(n, np.float32)
            np.add.at(g, gi[gi >= 0], d[gi >= 0])
            assert np.array_equal(g, np.array(wg, np.float32))


@pytest.mark.parametrize("seed", range(4))
def test_kernel_source_on_wide_frontiers(emu, gtn, seed):
    """Dense operands: levels of more than one chunk of the (emulated: 128-thread) CTA, parallel arcs racing for the
    same destination, and states with long arc lists, which whole warps enumerate (warp_out_arcs)."""
    rng = np.random.default_rng(40 + seed)
    a, b, intersect = case(rng, seed, 20, 110, 0.1)
    ma, mb = ours_from(gtn, a), ours_from(gtn, b)
    if seed & 1:
        ma.arc_sort(True)
    if seed & 2:
        mb.arc_sort(False)
    out = run(emu, gtn, ma, mb, intersect, cap=1 << 20, reach_ctas=1 + seed % 3)
    gtn.set_compose_device_policy(2)
    try:
        host = gtn.intersect(ma, mb) if intersect else gtn.compose(ma, mb)
    finally:
        gtn.set_compose_device_policy(0)
    check_against(out, ours_arrays(host), "vs the host construction")


def test_ngram_ctc_operands(emu, gtn):
    """intersect(ctc, transitions) of timeNgramCtc (benchmarks/ctc.cpp:60-80, 107-123): CTC target graph x dense
    bigram graph, both cyclic, both arc-sorted."""
    M, U = 30, 10
    rng = np.random.default_rng(1)
    target = rng.integers(1, M, U)
    ctc = gtn.Graph(False)
    L = 2 * U + 1
    for l in range(L):
        idx = (l - 1) // 2
        ctc.add_node(l == 0, l == L - 1 or l == L - 2)
        label = int(target[idx]) if l % 2 else 0
        ctc.add_arc(l, l, label)
        if l > 0:
            ctc.add_arc(l - 1, l, label)
        if l % 2 and l > 1 and label != int(target[idx - 1]):
            ctc.add_arc(l - 2, l, label)
    ctc.arc_sort()
    trans = gtn.Graph()
    for i in range(M):
        trans.add_node(True, True)
    for i in range(M):
        for m in range(M):
            trans.add_arc(i, m, m, m, float(rng.integers(-3, 4)))
    trans.arc_sort()
    out = run(emu, gtn, ctc, trans, True)
    gtn.set_compose_device_policy(2)
    try:
        host = gtn.intersect(ctc, trans)
    finally:
        gtn.set_compose_device_policy(0)
    check_against(out, ours_arrays(host), "ngram ctc")
    assert len(out["flags"]) > L
