"""Parity AT the BASELINE.json configurations, against the reference itself.

tests/golden/reference_configs.npz holds what the unmodified reference computed on the same seeded inputs
as the CUDA path, at the config's own T / C / U (a slice of its batch where the CPU needs seconds per
utterance); tests/golden/make_golden.py regenerates it.  Both are additionally judged against a float64
evaluation (oracle/f64.py): the CUDA result must be within tolerance of the reference AND at least as
close to the exact answer as the reference is (x2).  The fixture keeps the reference's losses, paths and
transition gradients whole; of its emission gradients it keeps the exact per-utterance error against
float64 and a sample of the values (make_golden.py: grad_sample).  Observed errors are written to
parity_observed.json (summarised in DESIGN.md "Tolerances").
"""
import json
import os

import numpy as np
import pytest

from tests import util

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _record(name, stats):
    d = os.path.join(ROOT, "gpurun_out")
    os.makedirs(d, exist_ok=True)
    p = os.path.join(d, "parity_observed.json")
    try:
        cur = json.load(open(p))
    except Exception:
        cur = {}
    cur[name] = stats
    json.dump(cur, open(p, "w"), indent=1, sort_keys=True)


@pytest.fixture(scope="module")
def ref():
    return util.golden_configs()


def _sampled(g, idx):
    return np.take_along_axis(g.reshape(len(idx), -1), idx, 1)


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.maximum(np.abs(a), np.abs(b)), 1e-30)))


@pytest.fixture(scope="module")
def c2(ref):
    """64 utterances of BASELINE configs[1] (the first 64 of bench.py's B=256 batch: seeds 1234+b),
    the reference's losses/gradients and the float64 referee's."""
    from oracle import f64
    n, T, C, U = 64, 1000, 64, 100
    e, tg = util.bench_inputs(n, T, C, U)
    lr = ref["ctc_loss"]
    gr = (ref["ctc_grad_idx"], ref["ctc_grad"], ref["ctc_grad_err_max"], ref["ctc_grad_err_mean"])
    l64 = np.zeros(n)
    g64 = np.zeros((n, T, C))
    for b in range(n):
        l64[b], g64[b] = f64.ctc_f64(e[b], tg[b])
    return e, tg, lr, gr, l64, g64


@pytest.mark.parametrize("buffers", ["device", "host"])
def test_ctc_config2_batch_vs_reference(ctx, c2, buffers):
    """configs[1]: CTC loss + gradient, T=1000 C=64 U=100, 64 utterances of the benchmark batch through
    gtnb_ctc_loss with device pointers (the `value` leg of bench.py) and with host buffers (the `e2e`
    leg).  Reference: benchmarks/ctc.cpp:150-165."""
    e, tg, lr, gr, l64, g64 = c2
    n, T, C = e.shape
    if buffers == "device":
        lo, go = ctx.ctc_loss_dev(e, tg)
    else:
        lo, go = ctx.ctc_loss(e, tg)
    assert np.all(np.isfinite(lo))
    # scores: north-star 1e-4 relative (observed ~1e-7)
    assert _rel(lo, lr) <= 1e-4
    assert _rel(lo, l64) <= 1e-4
    idx, gr_sample, ref_err, ref_mean_err = gr
    my_err = np.abs(go - g64).reshape(n, -1).max(axis=1)
    vs_ref = np.abs(_sampled(go, idx) - gr_sample).max(axis=1)
    _record("ctc_config2_%s" % buffers, {
        "n": n, "max_rel_loss_vs_ref": _rel(lo, lr), "max_rel_loss_vs_f64": _rel(lo, l64),
        "ref_max_rel_loss_vs_f64": _rel(lr, l64),
        "max_abs_grad_vs_ref": float(vs_ref.max()), "max_abs_grad_vs_f64": float(my_err.max()),
        "ref_max_abs_grad_vs_f64": float(ref_err.max()),
        "mean_abs_grad_vs_f64": float(np.abs(go - g64).mean()),
        "ref_mean_abs_grad_vs_f64": float(ref_mean_err.mean())})
    # every utterance at least as close to the exact gradient as the reference is (x2 + 1e-5)
    assert np.all(my_err <= 2.0 * ref_err + 1e-5), (my_err.max(), ref_err.max())
    # ... and therefore within 3x the reference's own error OF the reference (triangle inequality;
    # stated explicitly because it is the direct CUDA-vs-reference number, taken on the fixture's sample,
    # which holds each utterance's positions of largest reference error: observed 2.6e-3 max abs over the
    # whole gradient where the reference itself is 2.8e-3 from the exact gradient)
    assert np.all(vs_ref <= 3.0 * ref_err + 2e-5), (vs_ref.max(), ref_err.max())
    # the mean error must not be worse than the reference's either (observed 1.1e-5 vs 4.0e-5)
    assert np.abs(go - g64).mean() <= 1.5 * ref_mean_err.mean() + 1e-7


def test_asg_config3_vs_reference(ctx, ref):
    """configs[2]: ASG loss with learned transitions, T=500 C=64 U=50, 16 utterances of the B=128
    batch sharing one transitions graph; emission gradients and the accumulated transition gradient
    (test/criterion_test.cpp:244-305)."""
    from oracle import f64
    n, T, C, U = 16, 500, 64, 50
    rng = np.random.default_rng(41)
    e = rng.uniform(-5, 5, (n, T, C)).astype(np.float32)
    tw = rng.uniform(-5, 5, C + C * C).astype(np.float32)
    tg = [rng.integers(0, C, U).astype(np.int32) for _ in range(n)]
    lr, tgr, ref_err = ref["asg_loss"], ref["asg_tgrad"], ref["asg_grad_err_max"]
    lo, go, tgo = ctx.asg_loss(e, tw, tg)
    l64 = np.zeros(n)
    g64 = np.zeros((n, T, C))
    t64 = np.zeros(C + C * C)
    for b in range(n):
        l64[b], g64[b], t = f64.asg_f64(e[b], tw, tg[b])
        t64 += t
    assert _rel(lo, lr) <= 1e-4 and _rel(lo, l64) <= 1e-4
    my_err = np.abs(go - g64).reshape(n, -1).max(axis=1)
    ref_terr = float(np.abs(tgr - t64).max())
    my_terr = float(np.abs(tgo - t64).max())
    vs_ref = np.abs(_sampled(go, ref["asg_grad_idx"]) - ref["asg_grad"]).max(axis=1)
    _record("asg_config3", {
        "n": n, "max_rel_loss_vs_ref": _rel(lo, lr), "max_rel_loss_vs_f64": _rel(lo, l64),
        "max_abs_grad_vs_ref": float(vs_ref.max()), "max_abs_grad_vs_f64": float(my_err.max()),
        "ref_max_abs_grad_vs_f64": float(ref_err.max()),
        "max_abs_transgrad_vs_ref": float(np.abs(tgo - tgr).max()), "max_abs_transgrad_vs_f64": my_terr,
        "ref_max_abs_transgrad_vs_f64": ref_terr, "transgrad_scale": float(np.abs(t64).max())})
    assert np.all(my_err <= 2.0 * ref_err + 1e-5), (my_err.max(), ref_err.max())
    assert my_terr <= 2.0 * ref_terr + 1e-4 * n, (my_terr, ref_terr)
    assert np.all(vs_ref <= 3.0 * ref_err + 2e-5), (vs_ref.max(), ref_err.max())
    assert float(np.abs(tgo - tgr).max()) <= 3.0 * ref_terr + 2e-4 * n


def test_viterbi_config4_vs_reference(ctx, ref):
    """configs[3]: viterbiScore + viterbiPath over compose(emissions, transitions) at T=2000 C=128
    (test/criterion_test.cpp:328-344): 3 utterances (the real reference needs seconds and ~3 GB per
    utterance), one of them integer valued so that ties occur on most frames.  Paths and
    scores compared with ==."""
    n, T, C = 3, 2000, 128
    rng = np.random.default_rng(99)
    e = rng.uniform(-5, 5, (n, T, C)).astype(np.float32)
    e[2] = np.round(e[2])
    for tw, pr, sr in zip((rng.uniform(-5, 5, C + C * C).astype(np.float32),
                           np.round(rng.uniform(-3, 3, C + C * C)).astype(np.float32)),
                          ref["vit_paths"], ref["vit_scores"]):
        po, so = ctx.viterbi_dense(e, tw)
        assert np.array_equal(po, pr)
        assert np.array_equal(so, sr)
    _record("viterbi_config4", {"n": 2 * n, "paths_equal": True, "scores_equal": True})


def test_forced_alignment_config4_vs_reference(ctx, ref, oracle):
    """configs[3], second data point of SURVEY.md 8(d): viterbiPath(intersect(ctc, emissions)) at
    T=2000 C=128 U=200 through the lattice API, 8 utterances against the reference, two of them
    integer valued (exact ties: shortest.cpp:212-218 first-relaxed-wins).  =="""
    n, T, C, U = 8, 2000, 128, 200
    e, tg = util.bench_inputs(n, T, C, U, seed=777)
    e[6:] = np.round(e[6:])
    pr, sr = ref["fa_paths"], ref["fa_scores"]
    e_dev = ctx.to_device(e)
    views = [util.view_of(oracle.Graph.ctc(t, 0, True)) for t in tg]
    lat = ctx.compose_linear(views, [T] * n, C, e_dev, T * C)
    out = lat.viterbi_path(T)
    sc = lat.forward(tropical=True)
    lat.free()
    e_dev.free()
    assert np.array_equal(sc, sr)
    for b in range(n):
        assert np.array_equal(out["ilabels"][b], pr[b]), b
