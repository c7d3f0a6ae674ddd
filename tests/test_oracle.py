"""CPU tests: the C oracle against the committed golden vectors (made by the real
reference, tests/golden/make_golden.py) and against the reference's own known-answer
tests; plus against the reference's results on seeded random graphs (tests/golden/reference_host.json)."""
import numpy as np
import pytest

from tests import util
from oracle import pyoracle as po

GOLD = np.load(util.__file__.replace("util.py", "golden/reference_golden.npz"))


def test_ctc_known_answers_criterion_test():
    """test/criterion_test.cpp:56-180."""
    T, N = 3, 2
    e = np.log(np.maximum(np.array([1.0, 0.0, 0.0, 1.0, 1.0, 0.0], np.float32), 0)).reshape(T, N)
    with np.errstate(divide="ignore"):
        e = np.log(np.array([1.0, 0.0, 0.0, 1.0, 1.0, 0.0], np.float32)).reshape(T, N)
    ctc = po.Graph.ctc([0, 0], 1, False)
    s, _, _, _ = po.shortest_distance(po.compose(ctc, po.Graph.linear(T, N, e)))
    assert s == 0.0
    # case 2 (:72-83)
    T, N = 3, 4
    e = np.log(np.ones((T, N), np.float32))
    ctc = po.Graph.ctc([1, 2], N - 1, False)
    lat = po.compose(ctc, po.Graph.linear(T, N, e))
    s, _, _, _ = po.shortest_distance(lat)
    z, _, _, _ = po.shortest_distance(po.Graph.linear(T, N, e))
    assert abs(-(s - z) - (-np.log(0.25 ** 3 * 5))) < 1e-5


def test_ctc_golden_config1():
    e, tg = util.bench_inputs(1, 100, 28, 10)
    lo, go = po.ctc_loss(e[0], tg[0])
    assert util.close(lo, GOLD["c1_loss"][0], rtol=1e-6)
    assert np.abs(go - GOLD["c1_grad"][0]).max() < 1e-6


def test_ctc_golden_config2_one_utterance():
    e, tg = util.bench_inputs(1, 1000, 64, 100)
    lo, go = po.ctc_loss(e[0], tg[0])
    assert util.close(lo, GOLD["c2_loss"][0], rtol=1e-6)
    # same libm, same operation order -> (near) bit-identical to the reference
    assert np.abs(go - GOLD["c2_grad"][0]).max() < 1e-5
    assert abs(lo - float(GOLD["c2_loss_f64"])) < 1e-3 * abs(lo)


def test_asg_golden():
    e, tw, tg = GOLD["asg_e"], GOLD["asg_tw"], GOLD["asg_targets"]
    tsum = np.zeros_like(GOLD["asg_tgrad"])
    for b in range(e.shape[0]):
        lo, go, tgr = po.asg_loss(e[b], tw, tg[b])
        assert util.close(lo, GOLD["asg_loss"][b], rtol=1e-6)
        assert np.abs(go - GOLD["asg_grad"][b]).max() < 1e-6
        tsum += tgr
    assert np.abs(tsum - GOLD["asg_tgrad"]).max() < 1e-5


def test_asg_known_answer_criterion_test():
    """test/criterion_test.cpp:182-306, first utterance: loss 7.7417464 and emission grads."""
    N, T = 6, 5
    e = np.array([
        -0.4340, -0.0254, 0.3667, 0.4180, -0.3805, -0.1707, 0.1060, 0.3631,
        -0.1122, -0.3825, -0.0031, -0.3801, 0.0443, -0.3795, 0.3194, -0.3130,
        0.0094, 0.1560, 0.1252, 0.2877, 0.1997, -0.4554, 0.2774, -0.2526,
        -0.4001, -0.2402, 0.1295, 0.0172, 0.1805, -0.3299], np.float32).reshape(T, N)
    g_want = np.array([
        0.1060, 0.1595, -0.7639, 0.2485, 0.1118, 0.1380, 0.1915, -0.7524,
        0.1539, 0.1175, 0.1717, 0.1178, 0.1738, 0.1137, 0.2288, 0.1216,
        0.1678, -0.8057, 0.1766, -0.7923, 0.1902, 0.0988, 0.2056, 0.1210,
        0.1212, 0.1422, 0.2059, -0.8160, 0.2166, 0.1300], np.float32).reshape(T, N)
    lo, go, _ = po.asg_loss(e, np.zeros(N + N * N, np.float32), [2, 1, 5, 1, 3])
    assert abs(lo - 7.7417464256287) < 1e-3
    assert np.abs(go - g_want).max() < 1e-4


def test_viterbi_golden_ties():
    e, tw = GOLD["vit_e"], GOLD["vit_tw"]
    for b in range(e.shape[0]):
        p, s = po.viterbi_dense(e[b], tw)
        assert np.array_equal(p, GOLD["vit_paths"][b])
        assert s == GOLD["vit_scores"][b]
        p, s = po.viterbi_ctc(e[b], GOLD["fa_targets"][b])
        assert np.array_equal(p, GOLD["fa_paths"][b])
        assert s == GOLD["fa_scores"][b]


def test_asg_viterbi_known_answer():
    """test/criterion_test.cpp:308-345 -> {2, 1, 1, 0}."""
    e = np.array([0, 0, 7, 5, 4, 3, 5, 8, 5, 5, 4, 3], np.float32).reshape(4, 3)
    trans = np.array([0, 2, 0, 0, 0, 2, 2, 0, 0], np.float32)
    tw = np.concatenate([np.zeros(3, np.float32), trans])
    p, _ = po.viterbi_dense(e, tw)
    assert p.tolist() == [2, 1, 1, 0]


def test_forward_known_answers():
    """test/functions_test.cpp:231-389."""
    g = po.Graph.from_arrays([], [], [], [], [])
    assert po.shortest_distance(g)[0] == -np.inf
    lab = lambda n: np.zeros(n, np.int32)
    g = po.Graph.from_arrays([1, 0, 2], [0, 0, 0, 1, 1, 1], [1, 1, 1, 2, 2, 2], lab(6), lab(6),
                             [1, 2, 3, 1, 2, 3])
    assert abs(po.shortest_distance(g)[0] - 6.8152) < 1e-4
    for src, dst in ([0], [0]), ([0, 1, 1], [1, 2, 1]), ([0, 1, 2], [1, 2, 0]), ([0, 1], [2, 2]):
        flags = [3] if len(src) == 1 else [1, 0, 2]
        g = po.Graph.from_arrays(flags, src, dst, lab(len(src)), lab(len(src)))
        with pytest.raises(po.OracleError):
            po.shortest_distance(g)
    # viterbiScore known answer (:391-410): max path
    g = po.Graph.from_arrays([1, 0, 2], [0, 0, 0, 1, 1, 1], [1, 1, 1, 2, 2, 2], lab(6), lab(6),
                             [1, 2, 3, 1, 2, 3])
    assert po.shortest_distance(g, True)[0] == 6.0


def rand_graph(rng, n, eps):
    a = int(rng.integers(n, 3 * n))
    flags = np.zeros(n, np.uint8)
    flags[0] = 1
    flags[-1] = 2
    flags[int(rng.integers(0, n))] |= int(rng.integers(0, 4))
    src = rng.integers(0, n, a).astype(np.int32)
    dst = rng.integers(0, n, a).astype(np.int32)
    il = rng.integers(-1 if eps else 0, 3, a).astype(np.int32)
    ol = rng.integers(-1 if eps else 0, 3, a).astype(np.int32)
    w = rng.uniform(-1, 1, a).astype(np.float32)
    return flags, src, dst, il, ol, w


@pytest.mark.parametrize("seed", range(4))
def test_oracle_vs_live_reference_random(seed):
    """Exact structural equality of compose (all three matchers), scores, gradients, paths, against what the
    reference computed on the same seeded graphs (tests/golden/reference_host.json)."""
    gold = util.golden_host()["oracle"][str(seed)]
    want = iter(gold["compose"])
    rng = np.random.default_rng(100 + seed)
    for _ in range(10):
        n1, n2 = int(rng.integers(2, 8)), int(rng.integers(2, 8))
        eps = bool(rng.integers(0, 2))
        a1, a2 = rand_graph(rng, n1, eps), rand_graph(rng, n2, eps)
        g1, g2 = po.Graph.from_arrays(*a1), po.Graph.from_arrays(*a2)
        sort_mode = int(rng.integers(0, 4))
        if sort_mode & 1:
            g1.arc_sort(True)
        if sort_mode & 2:
            g2.arc_sort(False)
        for mode in (0, 1):
            mine = po.compose(g1, g2) if mode == 0 else po.intersect(g1, g2)
            ma, ra = mine.arrays(), util.graph_arrays(next(want))
            assert mine.num_nodes == len(ra["flags"]) and mine.num_arcs == len(ra["src"])
            for k in ("flags", "src", "dst", "ilabel", "olabel", "w"):
                assert np.array_equal(ma[k], ra[k]), k
    # DAGs: scores, gradients, best paths
    for dag in gold["dags"]:
        n = int(rng.integers(2, 30))
        arrs = util.random_dag(rng, n, int(rng.integers(n, 4 * n)), int_weights=bool(rng.integers(0, 2)))
        g = po.Graph.from_arrays(*arrs)
        for k, tropical in enumerate((False, True)):
            s, gr = po.forward_score_and_grad(g, tropical)
            assert util.close(s, dag["scores"][k], rtol=1e-6)
            rg = np.array(dag["grads"][k], np.float32)
            assert np.abs(rg - gr).max() < 1e-6
        path = po.shortest_path(g)
        assert np.array_equal(g.arrays()["ilabel"][path], np.array(dag["path_ilabel"], np.int32))
        assert np.array_equal(g.arrays()["w"][path], np.array(dag["path_w"], np.float32))
