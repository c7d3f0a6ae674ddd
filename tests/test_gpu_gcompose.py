"""General composition on the GPU (k_gcompose.cu through gtnb_compose_graphs and the gtn:: surface): arbitrary
operand pairs -- epsilons, cycles, any sortedness -- against the reference (its results on these seeded operands
stored in tests/golden/reference_host.json) and against the host construction: identical numbering, weights and
gradients."""
import numpy as np
import pytest

from tests import util
from tests.test_gcompose_emulation import case, check_against
from tests.test_host_api import golden, ours_arrays, ours_from, seed_like

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gtn():
    import gtn_b200.gtn as g
    return g


@pytest.fixture()
def on_device(gtn):
    gtn.set_compose_device_policy(1)
    yield
    gtn.set_compose_device_policy(0)


def host(gtn, fn, *args):
    gtn.set_compose_device_policy(2)
    try:
        return fn(*args)
    finally:
        gtn.set_compose_device_policy(1)


@pytest.mark.parametrize("seed", range(24))
def test_device_compose_matches_reference_numbering_and_gradients(gtn, on_device, seed):
    rng = np.random.default_rng(700 + seed)
    a, b, intersect = case(rng, seed, 7, 14, 0.2)
    ma, mb = ours_from(gtn, a), ours_from(gtn, b)
    if seed & 1:
        ma.arc_sort(True)
    if seed & 2:
        mb.arc_sort(False)
    before = gtn.device_launch_count()
    mo = gtn.intersect(ma, mb) if intersect else gtn.compose(ma, mb)
    assert gtn.device_launch_count() > before, "the device path did not run"
    ha, hb = ours_from(gtn, a), ours_from(gtn, b)
    if seed & 1:
        ha.arc_sort(True)
    if seed & 2:
        hb.arc_sort(False)
    ho = host(gtn, gtn.intersect if intersect else gtn.compose, ha, hb)
    check_against(ours_arrays(mo), ours_arrays(ho), "device vs host construction")
    want = golden("compose", seed)
    check_against(ours_arrays(mo), util.graph_arrays(want["out"]), "device vs reference")
    assert (want["grads"] is not None) == bool(mo.num_arcs())
    if mo.num_arcs():
        gtn.backward(mo, seed_like(gtn, mo, rng))
        for m, g in zip((ma, mb), want["grads"]):
            assert np.array_equal(np.array(m.grad().weights_to_list(), np.float32).reshape(-1), np.array(g, np.float32))


def test_list_overload_is_one_batched_call(gtn, on_device):
    rng = np.random.default_rng(5)
    As, Bs = [], []
    for s in range(12):
        a, b, _ = case(rng, 1, 30, 200, 0.15)
        ga, gb = ours_from(gtn, a), ours_from(gtn, b)
        if s & 1:
            ga.arc_sort(True)
        if s & 2:
            gb.arc_sort(False)
        As.append(ga)
        Bs.append(gb)
    before = gtn.device_launch_count()
    outs = gtn.compose(As, Bs)
    assert gtn.device_launch_count() - before <= 2, "12 pairs: one search and one fill launch"
    for ga, gb, o in zip(As, Bs, outs):
        check_against(ours_arrays(o), ours_arrays(host(gtn, gtn.compose, ga, gb)), "list entry")
    # a size-1 list broadcasts (parallel_map.h:77-89)
    outs = gtn.compose(As, [Bs[0]])
    for ga, o in zip(As, outs):
        check_against(ours_arrays(o), ours_arrays(host(gtn, gtn.compose, ga, Bs[0])), "broadcast entry")


def ctc_graph(gtn, target, blank=0):
    L = 2 * len(target) + 1
    g = gtn.Graph(False)
    for l in range(L):
        idx = (l - 1) // 2
        g.add_node(l == 0, l == L - 1 or l == L - 2)
        label = int(target[idx]) if l % 2 else blank
        g.add_arc(l, l, label)
        if l > 0:
            g.add_arc(l - 1, l, label)
        if l % 2 and l > 1 and label != int(target[idx - 1]):
            g.add_arc(l - 2, l, label)
    g.arc_sort()
    return g


def transitions_graph(gtn, M, N, rng):
    """benchmarks/ctc.cpp:60-80: M^(N-1) states, M arcs each"""
    n = M ** (N - 1)
    g = gtn.Graph()
    for _ in range(n):
        g.add_node(True, True)
    mod = max(n // M, 1)
    for i in range(n):
        for m in range(M):
            g.add_arc(i, (i % mod) * M + m if N > 2 else m, m, m, float(rng.uniform(-1, 1)))
    g.arc_sort()
    return g


def ngram_ctc_loss(gtn, ctc, emissions, transitions):
    num = gtn.forward_score(gtn.intersect(gtn.intersect(ctc, transitions), emissions))
    denom = gtn.forward_score(gtn.intersect(emissions, transitions))
    return gtn.subtract(denom, num)


def test_time_ngram_ctc_pipeline(gtn, on_device):
    """timeNgramCtc (benchmarks/ctc.cpp:107-134): intersect(ctc, transitions) on the device by k_gcompose.cu, the two
    intersections with the emissions by k_compose.cu; loss and all three gradients equal the host construction's."""
    T, U, M, N = 200, 10, 30, 2
    rng = np.random.default_rng(3)
    target = rng.integers(1, M, U)
    w = rng.uniform(-5, 5, (T, M)).astype(np.float32)

    def build():
        ctc = ctc_graph(gtn, target)
        em = gtn.linear_graph(T, M)
        em.set_weights(w.reshape(-1).tolist())
        tr = transitions_graph(gtn, M, N, np.random.default_rng(4))
        return ctc, em, tr

    ctc, em, tr = build()
    loss = ngram_ctc_loss(gtn, ctc, em, tr)
    gtn.backward(loss)
    hctc, hem, htr = build()
    hloss = host(gtn, ngram_ctc_loss, gtn, hctc, hem, htr)
    gtn.backward(hloss)
    assert loss.item() == pytest.approx(hloss.item(), rel=1e-6)
    for a, b in ((em, hem), (tr, htr)):
        ga = np.array(a.grad().weights_to_list(), np.float32)
        gb = np.array(b.grad().weights_to_list(), np.float32)
        assert np.allclose(ga, gb, rtol=1e-4, atol=1e-5)


def test_epsilon_operand_against_emissions(gtn):
    """An operand with epsilon arcs on the matched side composed with the emissions chain: not frame-synchronous
    (k_compose.cu declines), 1001 x N product states -> the general device path under the default policy."""
    T, C = 400, 8
    rng = np.random.default_rng(11)
    g = gtn.Graph()
    n = 48
    for i in range(n):
        g.add_node(i == 0, i == n - 1)
    for i in range(n - 1):
        g.add_arc(i, i + 1, int(rng.integers(0, C)), int(rng.integers(0, C)), float(rng.uniform(-1, 1)))
        g.add_arc(i, i, int(rng.integers(0, C)), int(rng.integers(0, C)), float(rng.uniform(-1, 1)))
        if i % 5 == 0:
            g.add_arc(i, i + 1, int(rng.integers(0, C)), gtn.epsilon, float(rng.uniform(-1, 1)))
    em = gtn.linear_graph(T, C)
    w = rng.uniform(-2, 2, T * C).astype(np.float32)
    em.set_weights(w.tolist())
    assert gtn.compose_device_policy() == 0
    before = gtn.device_launch_count()
    out = gtn.compose(g, em)
    assert gtn.device_launch_count() > before
    s = gtn.forward_score(out)
    gtn.backward(s)
    g2 = gtn.Graph()
    for i in range(n):
        g2.add_node(i == 0, i == n - 1)
    for a in range(g.num_arcs()):
        g2.add_arc(g.src_node(a), g.dst_node(a), g.ilabel(a), g.olabel(a), g.weight(a))
    em2 = gtn.linear_graph(T, C)
    em2.set_weights(w.tolist())
    gtn.set_compose_device_policy(2)
    try:
        out2 = gtn.compose(g2, em2)
    finally:
        gtn.set_compose_device_policy(0)
    check_against(ours_arrays(out), ours_arrays(out2), "epsilon operand x emissions")
    s2 = gtn.forward_score(out2)
    gtn.backward(s2)
    assert s.item() == pytest.approx(s2.item(), rel=1e-6)
    assert np.allclose(np.array(g.grad().weights_to_list()), np.array(g2.grad().weights_to_list()), rtol=1e-4, atol=1e-6)
    assert np.allclose(np.array(em.grad().weights_to_list()), np.array(em2.grad().weights_to_list()), rtol=1e-4, atol=1e-6)
