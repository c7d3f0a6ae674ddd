"""gtnb_ctc_align (k_align.cu, CTC forced alignment without the lattice) on the GPU: against the reference's
stored results at config 4, the lattice route (compose + exact-tie order + viterbi_path / tropical forward) and
the live reference (oracle/_ref) with ==; its fallback for non-finite emissions; the host / device / torch
entry points; edge cases and argument errors."""
import numpy as np
import pytest

from gtn_b200 import capi
from tests import util
from tests.test_align_emulation import check_states

pytestmark = pytest.mark.gpu


def lattice_route(ctx, oracle, e, targets, blank=0, arc_sorted=True, input_lens=None):
    """viterbiPath / viterbiScore through the lattice API: labels [B, T] (-1 padded), scores [B]."""
    B, T, C = e.shape
    lens = [T] * B if input_lens is None else [int(x) for x in input_lens]
    e_dev = ctx.to_device(e)
    views = [util.view_of(oracle.Graph.ctc(t, blank, arc_sorted)) for t in targets]
    lat = ctx.compose_linear(views, lens, C, e_dev, T * C)
    out = lat.viterbi_path(T)
    sc = lat.forward(tropical=True)
    lat.free()
    e_dev.free()
    labels = np.full((B, T), -1, np.int32)
    for b in range(B):
        n = int(out["lens"][b])
        labels[b, :max(n, 0)] = out["ilabels"][b, :max(n, 0)]
    return labels, sc


def reference(oracle, e, targets, blank, arc_sorted, input_lens):
    B, T, _ = e.shape
    labels = np.full((B, T), -1, np.int32)
    scores = np.zeros(B, np.float32)
    for b in range(B):
        Tb = T if input_lens is None else int(input_lens[b])
        p, s, _ = oracle.ref_viterbi_ctc_batch(e[b:b + 1, :Tb], [targets[b]], blank, arc_sorted)
        labels[b, :Tb] = p[0]
        scores[b] = s[0]
    return labels, scores


def check_batch(ctx, oracle, e, targets, blank=0, arc_sorted=True, input_lens=None):
    labels, scores, states = ctx.ctc_align(e, targets, blank, input_lens, arc_sorted, want_states=True)
    ll, ls = lattice_route(ctx, oracle, e, targets, blank, arc_sorted, input_lens)
    assert np.array_equal(labels, ll)
    assert np.array_equal(scores, ls)
    if oracle.have_ref():
        rl, rs = reference(oracle, e, targets, blank, arc_sorted, input_lens)
        assert np.array_equal(labels, rl)
        assert np.array_equal(scores, rs)
    T = e.shape[1]
    for b in range(len(targets)):
        check_states(labels[b], states[b], targets[b], blank, T if input_lens is None else int(input_lens[b]))
    return labels, scores, states


def test_forced_alignment_config4_vs_reference(ctx):
    """configs[3]'s forced alignment, 8 utterances at T=2000 C=128 U=200, two of them integer valued (ties on
    most frames): the reference's stored paths and scores, =="""
    n, T, C, U = 8, 2000, 128, 200
    e, tg = util.bench_inputs(n, T, C, U, seed=777)
    e[6:] = np.round(e[6:])
    ref = util.golden_configs()
    labels, scores, states = ctx.ctc_align_dev(e, tg, want_states=True)
    assert np.array_equal(labels, ref["fa_paths"])
    assert np.array_equal(scores, ref["fa_scores"])
    for b in range(n):
        check_states(labels[b], states[b], tg[b], 0, T)


@pytest.mark.parametrize("arc_sorted", [True, False])
def test_random_batches_vs_lattice_and_reference(ctx, oracle, arc_sorted):
    """Odd batch, ragged input and target lengths, U = 0, repeated labels, integer emissions, a blank inside the
    label range, an utterance too short for its target."""
    rng = np.random.default_rng(31 + arc_sorted)
    B, T, C = 7, 120, 20
    e = rng.uniform(-5, 5, (B, T, C)).astype(np.float32)
    e[1] = np.round(e[1])
    e[4] = rng.integers(-2, 3, (T, C)).astype(np.float32)
    tg = [rng.integers(1, C, U).astype(np.int32) for U in (30, 12, 0, 45, 20, 8, 40)]
    tg[3] = np.repeat(rng.integers(1, C, 15), 3).astype(np.int32)  # runs of repeated labels
    lens = np.array([120, 100, 7, 119, 60, 0, 50], np.int32)
    tg[6] = np.repeat(np.int32(5), 40)  # 40 repeats need 79 frames: no accepting path in 50
    check_batch(ctx, oracle, e, tg, 0, arc_sorted, lens)
    blank = 9
    tgb = [np.where(t == blank, 3, t).astype(np.int32) for t in tg]
    check_batch(ctx, oracle, e, tgb, blank, arc_sorted, None)


def test_nonfinite_emissions_take_the_lattice_route(ctx, oracle):
    """-inf and NaN on lattice arcs of some utterances: those are computed on the lattice route (the reference's
    inf / NaN propagation), the others are unchanged."""
    B, T, C, U = 6, 80, 16, 15
    e, tg = util.bench_inputs(B, T, C, U, seed=55)
    clean = ctx.ctc_align(e, tg, want_states=True)
    e[1, 10, :] = -np.inf
    e[3, 20, tg[3][0]] = np.nan
    e[4, :, 0] = -np.inf  # every blank arc: the path has to avoid blanks
    labels, scores, states = check_batch(ctx, oracle, e, tg)
    for b in (0, 2, 5):
        assert np.array_equal(labels[b], clean[0][b]) and scores[b] == clean[1][b]
        assert np.array_equal(states[b], clean[2][b])
    assert np.isneginf(scores[1])


def test_host_and_device_buffers_agree(ctx):
    e, tg = util.bench_inputs(9, 300, 32, 40, seed=3)
    lens = np.array([300, 299, 150, 81, 300, 0, 200, 299, 120], np.int32)
    h = ctx.ctc_align(e, tg, input_lens=lens, want_states=True)
    d = ctx.ctc_align_dev(e, tg, input_lens=lens, want_states=True)
    for a, b in zip(h, d):
        assert np.array_equal(a, b)
    for sorted_ in (True, False):
        a = ctx.ctc_align(e, tg, arc_sorted=sorted_)
        b = ctx.ctc_align_dev(e, tg, arc_sorted=sorted_)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2] is None and b[2] is None


def test_torch_entry_on_a_side_stream(ctx):
    torch = pytest.importorskip("torch")
    from gtn_b200 import torch_loss
    e, tg = util.bench_inputs(5, 400, 40, 60, seed=11)
    lens = np.array([400, 333, 399, 200, 400], np.int32)
    want = ctx.ctc_align(e, tg, input_lens=lens, arc_sorted=False, want_states=True)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        et = torch.from_numpy(e).cuda()
        labels, states, scores = torch_loss.ctc_align(et, tg, torch.from_numpy(lens), arc_sorted=False)
    s.synchronize()
    assert labels.dtype == torch.int32 and states.dtype == torch.int32 and scores.dtype == torch.float32
    assert labels.is_cuda and states.is_cuda and scores.is_cuda
    assert np.array_equal(labels.cpu().numpy(), want[0])
    assert np.array_equal(scores.cpu().numpy(), want[1])
    assert np.array_equal(states.cpu().numpy(), want[2])


def test_empty_batches_and_bad_arguments(ctx):
    lab, sc, st = ctx.ctc_align(np.zeros((0, 5, 4), np.float32), [], want_states=True)
    assert lab.shape == (0, 5) and sc.shape == (0,)
    lab, sc, st = ctx.ctc_align(np.zeros((3, 0, 4), np.float32), [[], [1], []], want_states=True)
    assert lab.shape == (3, 0) and list(sc) == [0.0, -np.inf, 0.0]
    e = np.zeros((2, 6, 4), np.float32)
    lib = capi.lib()
    with pytest.raises(capi.GtnbInvalidArgument):
        ctx.ctc_align(e, [[1], [1]], input_lens=[6, 7])
    with pytest.raises(capi.GtnbInvalidArgument):
        ctx.ctc_align(e, [[1], [1]], input_lens=[-1, 6])
    lens = np.array([1, -1], np.int32)
    out = np.zeros((2, 6), np.int32)
    scores = np.zeros(2, np.float32)
    cat = np.array([1], np.int32)
    rc = lib.gtnb_ctc_align(ctx.h, 2, 6, 4, e.ctypes.data, 0, None, cat.ctypes.data_as(capi._i32p),
                            lens.ctypes.data_as(capi._i32p), 0, 1, out.ctypes.data, None, 0,
                            scores.ctypes.data_as(capi._f32p))
    assert rc == capi.ERR_INVALID_ARGUMENT
    lens = np.array([1, 0], np.int32)
    rc = lib.gtnb_ctc_align(ctx.h, 2, 6, 4, e.ctypes.data, 0, None, None, lens.ctypes.data_as(capi._i32p), 0, 1,
                            out.ctypes.data, None, 0, scores.ctypes.data_as(capi._f32p))
    assert rc == capi.ERR_INVALID_ARGUMENT
    # a sorted CTC graph whose nodes have more out-arcs than C: the reference's matcher order is not reproduced
    with pytest.raises(capi.GtnbError) as ex:
        ctx.ctc_align(np.zeros((1, 6, 2), np.float32), [[1, 0, 1]], blank=0)
    assert ex.value.code == capi.ERR_UNSUPPORTED
    # ... while the insertion-order graph is fine there
    ctx.ctc_align(np.zeros((1, 6, 2), np.float32), [[1, 0, 1]], blank=0, arc_sorted=False)


def test_symbol_exported():
    assert hasattr(capi.lib(), "gtnb_ctc_align")
    assert "gtnb_ctc_align" in [s[0] for s in capi.SYMBOLS]
