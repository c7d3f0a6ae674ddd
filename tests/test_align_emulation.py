"""The SOURCE of gtn_b200/csrc/k_align.cu (CTC forced alignment on the implicit lattice: viterbiPath /
viterbiScore of intersect(ctcGraph(target), emissions) without building it) run on the CPU through the SIMT
emulator of tests/emu, against the oracle and, where it is built, the reference itself: paths with ==,
scores bit for bit, ties included."""
import ctypes as C
import os

import numpy as np
import pytest

from tests import emu_build, util

HERE = os.path.dirname(os.path.abspath(__file__))
f32p, i32p = C.POINTER(C.c_float), C.POINTER(C.c_int32)
GOLD = np.load(os.path.join(HERE, "golden", "reference_golden.npz"))


@pytest.fixture(scope="module")
def emu():
    lib = C.CDLL(emu_build.build("align", ["k_align.cu"]))
    lib.emu_ctc_align.argtypes = [C.c_int, C.c_int, C.c_int, f32p, i32p, i32p, i32p, C.c_int, C.c_int, C.c_int,
                                  i32p, i32p, f32p, i32p]
    return lib


def run(emu, e, targets, blank=0, arc_sorted=True, input_lens=None, threads=0):
    e = np.ascontiguousarray(e, np.float32)
    B, T, Cn = e.shape
    lens = np.asarray([len(t) for t in targets], np.int32)
    cat = np.ascontiguousarray(np.concatenate([np.asarray(t, np.int32) for t in targets] + [np.zeros(1, np.int32)]))
    il = None if input_lens is None else np.ascontiguousarray(input_lens, np.int32)
    labels = np.full((B, max(T, 1)), -7, np.int32)
    states = np.full_like(labels, -7)
    scores = np.full(B, 7.0, np.float32)
    status = np.full(B, -7, np.int32)
    rc = emu.emu_ctc_align(B, T, Cn, e.ctypes.data_as(f32p), None if il is None else il.ctypes.data_as(i32p),
                           cat.ctypes.data_as(i32p), lens.ctypes.data_as(i32p), blank, int(arc_sorted), threads,
                           labels.ctypes.data_as(i32p), states.ctypes.data_as(i32p), scores.ctypes.data_as(f32p),
                           status.ctypes.data_as(i32p))
    emu_build.check(rc)
    return labels[:, :T], states[:, :T], scores, status


def check_states(lab, st, target, blank, Tb):
    """states is a CTC path that emits lab: starts in node 0 / 1, moves by self / step / skip, ends accepting."""
    L = 2 * len(target) + 1
    if Tb == 0 or lab[0] < 0:
        assert np.all(st == -1) and np.all(lab == -1)
        return
    assert np.all(st[Tb:] == -1) and np.all(lab[Tb:] == -1)
    s = st[:Tb]
    assert s[0] in (0, 1) and s[-1] in (L - 1, L - 2)
    d = np.diff(s)
    assert np.all((d >= 0) & (d <= 2))
    for t in np.nonzero(d == 2)[0]:  # a skip: between two different labels
        assert s[t] % 2 == 1 and target[s[t] // 2] != target[s[t] // 2 + 1]
    y = np.append(np.asarray(target, np.int64), -1)  # (the -1 pads U = 0)
    want = np.where(s % 2 == 1, y[np.maximum(s - 1, 0) // 2], blank)
    assert np.array_equal(lab[:Tb], want)


def check_vs_oracle(oracle, e, targets, got, blank=0, arc_sorted=True, input_lens=None):
    labels, states, scores, status = got
    B, T, _ = e.shape
    for b in range(B):
        Tb = T if input_lens is None else int(input_lens[b])
        assert status[b] == 0, b
        want_path, want_score = oracle.viterbi_ctc(e[b, :Tb], targets[b], blank, arc_sorted)
        assert np.array_equal(labels[b, :Tb], want_path), (b, labels[b, :Tb], want_path)
        assert np.all(labels[b, Tb:] == -1)
        assert scores[b] == np.float32(want_score), (b, scores[b], want_score)
        check_states(labels[b], states[b], targets[b], blank, Tb)


def test_golden_forced_alignment(emu, oracle):
    """tests/golden fa_*: what the reference computed (T=30, C=6, integer scores: ties on most frames)."""
    e, tg = GOLD["vit_e"], list(GOLD["fa_targets"])
    labels, states, scores, status = got = run(emu, e, tg)
    assert np.all(status == 0)
    assert np.array_equal(labels, GOLD["fa_paths"])
    assert np.array_equal(scores, GOLD["fa_scores"])
    check_vs_oracle(oracle, e, tg, got)


@pytest.mark.parametrize("arc_sorted", [True, False])
@pytest.mark.parametrize("blank", [0, 3, 7])
def test_integer_emissions_ties(emu, oracle, arc_sorted, blank):
    """Small integer scores: equal-score paths everywhere, the first-relaxed predecessor must win under both
    out-arc orders; a blank in the middle of the label range makes the sorted order differ from insertion."""
    rng = np.random.default_rng(10 * blank + arc_sorted)
    B, T, Cn = 4, 40, 8
    e = rng.integers(-2, 3, (B, T, Cn)).astype(np.float32)
    tg = [rng.integers(0, Cn, U).astype(np.int32) for U in (3, 7, 12, 1)]
    tg = [np.where(t == blank, (blank + 1) % Cn, t).astype(np.int32) for t in tg]
    got = run(emu, e, tg, blank=blank, arc_sorted=arc_sorted)
    check_vs_oracle(oracle, e, tg, got, blank, arc_sorted)
    if oracle.have_ref():
        pr, sr, _ = oracle.ref_viterbi_ctc_batch(e, tg, blank, arc_sorted)
        assert np.array_equal(got[0], pr) and np.array_equal(got[2], sr)


def test_repeats_and_tiny_graphs(emu, oracle):
    """Repeated labels (no skip arcs), U = 0, U = 1, and a target that needs every frame."""
    rng = np.random.default_rng(5)
    T, Cn = 9, 5
    e = rng.uniform(-5, 5, (6, T, Cn)).astype(np.float32)
    tg = [np.array([2, 2, 2], np.int32), np.zeros(0, np.int32), np.array([4], np.int32),
          np.array([1, 1, 3, 3], np.int32), np.array([1, 2, 1, 2, 3], np.int32), np.array([3, 3, 3, 3], np.int32)]
    for arc_sorted in (True, False):
        check_vs_oracle(oracle, e, tg, run(emu, e, tg, arc_sorted=arc_sorted), 0, arc_sorted)
    e1 = rng.uniform(-5, 5, (3, 1, Cn)).astype(np.float32)  # T = 1
    tg1 = [np.zeros(0, np.int32), np.array([2], np.int32), np.array([2, 3], np.int32)]
    check_vs_oracle(oracle, e1, tg1, run(emu, e1, tg1))


def test_no_path_and_ragged(emu, oracle):
    """Ragged input_lens and target lengths, T_b = 0, and utterances too short for their targets (no accepting
    path: labels -1, score -inf)."""
    rng = np.random.default_rng(6)
    B, T, Cn = 7, 16, 6
    e = rng.uniform(-5, 5, (B, T, Cn)).astype(np.float32)
    e[3] = np.round(e[3])
    tg = [rng.integers(1, Cn, U).astype(np.int32) for U in (4, 0, 9, 5, 2, 3, 6)]
    tg[4] = np.array([2, 2], np.int32)  # needs 3 frames
    lens = np.array([16, 0, 11, 13, 2, 0, 5], np.int32)
    labels, states, scores, status = got = run(emu, e, tg, input_lens=lens)
    check_vs_oracle(oracle, e, tg, got, input_lens=lens)
    assert scores[1] == 0.0 and np.isneginf(scores[4]) and np.isneginf(scores[5])
    assert np.all(labels[4] == -1) and np.all(states[5] == -1)


@pytest.mark.parametrize("threads", [64, 96])
def test_several_nodes_per_thread(emu, oracle, threads):
    """Graphs wider than the block: 2U+1 = 121 nodes over 64 threads (2 nodes per thread) and 96 (2 with a
    tail), plus the one-node-per-thread layout on the same inputs."""
    rng = np.random.default_rng(threads)
    B, T, Cn = 2, 150, 12
    e = rng.integers(-2, 3, (B, T, Cn)).astype(np.float32)
    tg = [rng.integers(1, Cn, 60).astype(np.int32), rng.integers(1, 4, 45).astype(np.int32)]
    for arc_sorted in (True, False):
        got = run(emu, e, tg, arc_sorted=arc_sorted, threads=threads)
        check_vs_oracle(oracle, e, tg, got, 0, arc_sorted)
        base = run(emu, e, tg, arc_sorted=arc_sorted)
        for a, b in zip(got, base):
            assert np.array_equal(a, b)


def test_out_of_envelope_status(emu):
    """A non-finite weight on a lattice arc (inf, -inf, NaN) or a label outside [0, C) marks the utterance for
    the lattice route; the others are computed as usual.  A non-finite emission no arc reads is harmless."""
    rng = np.random.default_rng(8)
    B, T, Cn = 6, 12, 5
    e = rng.uniform(-5, 5, (B, T, Cn)).astype(np.float32)
    tg = [np.array([1, 2, 3], np.int32)] * 4 + [np.array([1, 9], np.int32), np.array([1, 2], np.int32)]
    e[0, 4, 0] = np.inf
    e[1, 7, :] = -np.inf
    e[2, 0, 0] = np.nan
    e[3, 5, 4] = np.nan  # label 4 is in no target: never read
    labels, states, scores, status = run(emu, e, tg)
    assert list(status) == [1, 1, 1, 0, 2, 0]
    ref = run(emu, np.delete(e, [0, 1, 2, 4], 0), [tg[3], tg[5]])
    assert np.array_equal(labels[[3, 5]], ref[0]) and np.array_equal(scores[[3, 5]], ref[2])
    assert list(run(emu, e[3:4], [tg[3]], blank=Cn)[3]) == [2]  # blank outside [0, C)


def test_matches_bench_inputs(emu, oracle):
    """The benchmark's input distribution (util.bench_inputs) at a reduced size, float scores."""
    e, tg = util.bench_inputs(3, 60, 16, 12, seed=777)
    e[2] = np.round(e[2])
    for arc_sorted in (True, False):
        check_vs_oracle(oracle, e, tg, run(emu, e, tg, arc_sorted=arc_sorted), 0, arc_sorted)
