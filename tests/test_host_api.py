"""Host side of the gtn:: surface (SURVEY.md section 8(f) ranks 3-4): the rational operations, graph
comparison, the two wire formats, Graphviz export and random sampling of gtn_b200.gtn against

  * what the UNMODIFIED reference computed on the same seeded random graphs (tests/golden/reference_host.json,
    made by tests/golden/make_golden.py; outputs compared node by node and arc by arc, byte by byte for the
    wire formats), and
  * hand-derived known answers.

None of this touches the GPU: these functions are graph construction / tooling, exactly as in the
reference (gtn/functions.cpp:93-223,253-318; gtn/utils.cpp; gtn/rand.cpp)."""
import os

import numpy as np
import pytest

from tests import util


@pytest.fixture(scope="module")
def gtn():
    import gtn_b200.gtn as g
    return g


# ---------------------------------------------------------------------------------------------
# helpers


def random_graph(rng, n_nodes, n_arcs, n_labels=3, p_eps=0.25, transducer=True, int_weights=True):
    """Arbitrary graph: cycles, self-loops, parallel arcs, epsilons, several start / accept nodes."""
    flags = np.zeros(n_nodes, np.uint8)
    flags[rng.integers(0, n_nodes, max(1, n_nodes // 3))] |= 1
    flags[rng.integers(0, n_nodes, max(1, n_nodes // 3))] |= 2
    src = rng.integers(0, n_nodes, n_arcs).astype(np.int32)
    dst = rng.integers(0, n_nodes, n_arcs).astype(np.int32)
    il = rng.integers(0, n_labels, n_arcs).astype(np.int32)
    ol = rng.integers(0, n_labels, n_arcs).astype(np.int32) if transducer else il.copy()
    eps = rng.random(n_arcs) < p_eps
    il[eps] = -1
    ol[eps & (rng.random(n_arcs) < 0.7)] = -1
    w = (rng.integers(-4, 5, n_arcs) if int_weights else rng.uniform(-3, 3, n_arcs)).astype(np.float32)
    return flags, src, dst, il, ol, w


def ours_from(gtn, arrs, calc_grad=True):
    flags, src, dst, il, ol, w = arrs
    g = gtn.Graph(calc_grad)
    for f in flags:
        g.add_node(bool(f & 1), bool(f & 2))
    for a in range(len(src)):
        g.add_arc(int(src[a]), int(dst[a]), int(il[a]), int(ol[a]), float(w[a]))
    return g


def ours_arrays(g):
    n, a = g.num_nodes(), g.num_arcs()
    flags = np.array([(1 if g.is_start(i) else 0) | (2 if g.is_accept(i) else 0) for i in range(n)], np.uint8)
    return dict(flags=flags,
                src=np.array([g.src_node(i) for i in range(a)], np.int32),
                dst=np.array([g.dst_node(i) for i in range(a)], np.int32),
                ilabel=np.array([g.ilabel(i) for i in range(a)], np.int32),
                olabel=np.array([g.olabel(i) for i in range(a)], np.int32),
                w=np.array(g.weights_to_list(), np.float32).reshape(-1))


def assert_same(ours, want, what=""):
    """Identical numbering: node flags and the arc list, in order.  want: a graph of the golden fixture."""
    o, r = ours_arrays(ours), util.graph_arrays(want)
    for k in ("flags", "src", "dst", "ilabel", "olabel", "w"):
        assert o[k].shape == r[k].shape, (what, k, o[k].shape, r[k].shape)
        assert np.array_equal(o[k], r[k]), (what, k, o[k], r[k])


def seed_like(gtn, out_ours, rng):
    """Random deltas for backward(g, grad): same arc count as the output."""
    a = ours_arrays(out_ours)
    d = rng.integers(-5, 6, len(a["src"])).astype(np.float32)
    return ours_from(gtn, (a["flags"], a["src"], a["dst"], a["ilabel"], a["olabel"], d), calc_grad=False)


def golden(test, seed):
    return util.golden_host()[test][str(seed)]


# ---------------------------------------------------------------------------------------------
# rational operations against the reference


@pytest.mark.parametrize("seed", range(6))
def test_concat_closure_union_match_reference(gtn, seed):
    rng = np.random.default_rng(100 + seed)
    graphs = [random_graph(rng, int(rng.integers(1, 7)), int(rng.integers(0, 12))) for _ in range(4)]
    mine = [ours_from(gtn, g) for g in graphs]
    want = iter(golden("concat", seed))

    for k in range(0, 5):
        assert_same(gtn.concat(mine[:k]), next(want), "concat of %d" % k)
        assert_same(gtn.union(mine[:k]), next(want), "union of %d" % k)
    assert_same(gtn.concat(mine[0], mine[1]), next(want), "binary concat")
    for m in mine:
        assert_same(gtn.closure(m), next(want), "closure")
        clones = [next(want) for _ in range(3)]
        for proj, name in ((0, gtn.Projection.NONE), (1, gtn.Projection.INPUT), (2, gtn.Projection.OUTPUT)):
            assert_same(gtn.clone(m, name), clones[proj], "clone %d" % proj)
        assert_same(gtn.project_input(m), clones[1])
        assert_same(gtn.project_output(m), clones[2])


@pytest.mark.parametrize("seed", range(8))
def test_remove_matches_reference(gtn, seed):
    rng = np.random.default_rng(200 + seed)
    arrs = random_graph(rng, int(rng.integers(2, 9)), int(rng.integers(1, 20)), p_eps=0.4)
    m = ours_from(gtn, arrs)
    want = golden("remove", seed)
    assert_same(gtn.remove(m), want[0], "remove epsilon")
    assert_same(gtn.remove(m, 1), want[1], "remove label 1")
    assert_same(gtn.remove(m, -1, 1), want[2], "remove eps:1")
    assert_same(gtn.remove(m, 0, 2), want[3], "remove 0:2")
    # list overload (bindings/python/gtn/_functions.cpp:195-203): labels broadcast
    for got in gtn.remove([m, m]):
        assert_same(got, want[0], "remove list")


@pytest.mark.parametrize("seed", range(4))
def test_rational_gradients_match_reference(gtn, seed):
    """gradFuncs slice `deltas` by arc position (functions.cpp:98-110,158-163,193-202)."""
    rng = np.random.default_rng(300 + seed)
    graphs = [random_graph(rng, int(rng.integers(1, 6)), int(rng.integers(1, 9))) for _ in range(3)]
    for op_ours, want in zip((gtn.concat, gtn.union, lambda gs: gtn.closure(gs[0])), golden("rational_grads", seed)):
        mine = [ours_from(gtn, g, calc_grad=(i != 1)) for i, g in enumerate(graphs)]
        out_m = op_ours(mine)
        gtn.backward(out_m, seed_like(gtn, out_m, rng))
        used = 1 if op_ours not in (gtn.concat, gtn.union) else len(mine)
        assert len(want) == used
        for i in range(used):
            if i == 1 and used > 1:
                assert not mine[i].is_grad_available()
                continue
            assert np.array_equal(np.array(mine[i].grad().weights_to_list(), np.float32).reshape(-1),
                                  np.array(want[i], np.float32)), (i, op_ours)


def test_remove_has_no_gradient(gtn):
    g = gtn.Graph()
    g.add_node(True)
    g.add_node(False, True)
    g.add_arc(0, 1, gtn.epsilon)
    with pytest.raises(RuntimeError):  # std::logic_error (functions.cpp:273-275)
        gtn.backward(gtn.remove(g))


# ---------------------------------------------------------------------------------------------
# known answers that need no reference


def test_concat_known_answers(gtn):
    # a^0: one node, start and accept
    e = gtn.concat([])
    assert (e.num_nodes(), e.num_arcs(), e.is_start(0), e.is_accept(0)) == (1, 0, True, True)
    # "ab" . "c": accept of the first joined to the start of the second by one epsilon arc
    a = gtn.Graph()
    for i in range(3):
        a.add_node(i == 0, i == 2)
    a.add_arc(0, 1, 0)
    a.add_arc(1, 2, 1)
    b = gtn.Graph()
    b.add_node(True)
    b.add_node(False, True)
    b.add_arc(0, 1, 2, 5, 1.5)
    c = gtn.concat(a, b)
    assert gtn.dumps(c) == "0\n4\n0 1 0 0 0\n1 2 1 1 0\n3 4 2 5 1.5\n2 3 -1 -1 0\n"


def test_closure_and_union_known_answers(gtn):
    a = gtn.Graph()
    a.add_node(True)
    a.add_node(False, True)
    a.add_arc(0, 1, 7, 8, 0.25)
    # closure: new node 0 (start + accept), old nodes shifted by one, eps in and eps back
    assert gtn.dumps(gtn.closure(a)) == "0\n0\n1 2 7 8 0.25\n0 1 -1 -1 0\n2 0 -1 -1 0\n"
    u = gtn.union([a, a])
    assert gtn.dumps(u) == "0 2\n1 3\n0 1 7 8 0.25\n2 3 7 8 0.25\n"
    assert gtn.union([]).num_nodes() == 0


def test_remove_known_answer(gtn):
    # 0 -eps-> 1 -a-> 2(accept), 0 -b-> 2: node 1 is only reachable through epsilon and disappears
    g = gtn.Graph()
    g.add_node(True)
    g.add_node()
    g.add_node(False, True)
    g.add_arc(0, 1, gtn.epsilon)
    g.add_arc(1, 2, 4)
    g.add_arc(0, 2, 5)
    r = gtn.remove(g)
    assert gtn.dumps(r) == "0\n1\n0 1 5 5 0\n0 1 4 4 0\n"
    # an epsilon straight into an accept node makes the source accepting
    h = gtn.Graph()
    h.add_node(True)
    h.add_node(False, True)
    h.add_arc(0, 1, gtn.epsilon)
    r = gtn.remove(h)
    assert (r.num_nodes(), r.num_arcs(), r.is_start(0), r.is_accept(0)) == (1, 0, True, True)


# ---------------------------------------------------------------------------------------------
# comparison


@pytest.mark.parametrize("seed", range(10))
def test_equal_and_isomorphic_agree_with_reference(gtn, seed):
    rng = np.random.default_rng(400 + seed)
    n = int(rng.integers(1, 8))
    flags, src, dst, il, ol, w = random_graph(rng, n, int(rng.integers(0, 14)), n_labels=2, p_eps=0.1)
    base = (flags, src, dst, il, ol, w)
    # (a) the same graph with nodes renumbered and arcs shuffled, (b) one arc perturbed
    perm = rng.permutation(n)
    order = rng.permutation(len(src))
    renum = (flags[np.argsort(perm)], perm[src][order].astype(np.int32), perm[dst][order].astype(np.int32),
             il[order], ol[order], w[order])
    shuf = (flags, src[order], dst[order], il[order], ol[order], w[order])
    variants = [base, renum, shuf]
    if len(src):
        w2 = w.copy()
        w2[0] += 1.0
        variants.append((flags, src, dst, il, ol, w2))
        d2 = dst.copy()
        d2[-1] = (d2[-1] + 1) % n
        variants.append((flags, src, d2, il, ol, w))
    f2 = flags.copy()
    f2[0] ^= 2
    variants.append((f2, src, dst, il, ol, w))
    m0 = ours_from(gtn, base)
    want = golden("equal", seed)
    assert len(want) == len(variants)
    for k, (v, (equal, isomorphic)) in enumerate(zip(variants, want)):
        m = ours_from(gtn, v)
        assert gtn.equal(m0, m) == equal, ("equal", k)
        assert gtn.isomorphic(m0, m) == isomorphic, ("isomorphic", k)
    assert gtn.equal(m0, ours_from(gtn, shuf)) and gtn.isomorphic(m0, ours_from(gtn, shuf))


def test_isomorphic_known_answers(gtn):
    def chain(labels, loop_at=None):
        g = gtn.Graph()
        g.add_node(True)
        for i, l in enumerate(labels):
            g.add_node(False, i + 1 == len(labels))
            g.add_arc(i, i + 1, l)
        if loop_at is not None:
            g.add_arc(loop_at, loop_at, 9)
        return g

    assert gtn.isomorphic(chain([1, 2, 3]), chain([1, 2, 3]))
    assert not gtn.isomorphic(chain([1, 2, 3]), chain([1, 3, 2]))
    assert not gtn.isomorphic(chain([1, 2], loop_at=0), chain([1, 2], loop_at=1))
    # a cycle: 0 -> 1 -> 0 numbered the other way round
    a = gtn.Graph()
    a.add_node(True, True)
    a.add_node()
    a.add_arc(0, 1, 1)
    a.add_arc(1, 0, 2)
    b = gtn.Graph()
    b.add_node()
    b.add_node(True, True)
    b.add_arc(1, 0, 1)
    b.add_arc(0, 1, 2)
    assert gtn.isomorphic(a, b) and not gtn.equal(a, b)


# ---------------------------------------------------------------------------------------------
# wire formats


@pytest.mark.parametrize("seed", range(5))
def test_wire_formats_are_byte_compatible_with_reference(gtn, seed, tmp_path):
    rng = np.random.default_rng(500 + seed)
    n_arcs = int(rng.integers(0, 40))
    arrs = random_graph(rng, int(rng.integers(1, 30)), n_arcs, int_weights=(seed % 2 == 0))
    m = ours_from(gtn, arrs)
    want = golden("wire", seed)
    ref_bin, ref_txt = bytes.fromhex(want["bin"]), want["txt"].encode()
    # what we write is what the reference writes
    assert gtn.dumpb(m) == ref_bin
    assert gtn.dumps(m).encode() == ref_txt
    assert repr(m) == want["repr"]  # abbreviated above 20 nodes / arcs
    dot = str(tmp_path / "g.dot")
    gtn.write_dot(m, dot)
    assert open(dot, "rb").read() == want["dot"].encode("utf-8")
    # what either writes, the other reads (our bytes are the reference's, asserted above)
    assert_same(gtn.loadb(ref_bin), want["graph"], "ours reads the reference's binary")
    assert_same(m, want["from_bin"], "the reference reads our binary")
    assert ("from_txt" in want) == bool(arrs[0].any() and (arrs[0] & 2).any())
    if "from_txt" in want:  # the text format needs a start and an accept node
        assert gtn.equal(gtn.loads(ref_txt.decode()), gtn.loads(gtn.dumps(m)))
        assert_same(gtn.loads(gtn.dumps(m)), want["from_txt"], "text round trip through both parsers")
    # files
    fb, ft = str(tmp_path / "g.bin"), str(tmp_path / "g.txt")
    gtn.save(fb, m)
    assert open(fb, "rb").read() == ref_bin
    assert gtn.equal(gtn.load(fb), m)
    gtn.savetxt(ft, m)
    assert open(ft, "rb").read() == ref_txt


def test_write_dot_with_symbols(gtn, tmp_path):
    g = gtn.Graph()
    g.add_node(True)
    g.add_node(False, True)
    g.add_arc(0, 1, 0, 1, 0.5)
    g.add_arc(0, 1, gtn.epsilon, 0, 0.0)
    p = str(tmp_path / "s.dot")
    gtn.write_dot(g, p, {0: "a", 1: "b"}, {0: "x", 1: "y"})
    txt = open(p, encoding="utf-8").read()
    assert txt.startswith("digraph FST {") and txt.endswith("}")
    assert '0 -> 1 [label = "a:y/0.5"' in txt and '0 -> 1 [label = "ε:x/0"' in txt
    assert "doublecircle" in txt and "penwidth = 2.0" in txt
    with pytest.raises(RuntimeError):
        gtn.write_dot(g, os.path.join(str(tmp_path), "no", "such", "dir", "x.dot"))


def test_text_format_known_answers_and_errors(gtn, tmp_path):
    # the cases test/utils_test.cpp:348-432 pins
    g = gtn.loads("0\n0 1\n0 0 1 1 0\n0 2 1 1 1.1\n2 1 2 2 2.1\n")
    assert (g.num_nodes(), g.num_arcs()) == (3, 3)
    assert g.is_start(0) and g.is_accept(0) and g.is_accept(1) and not g.is_accept(2)
    assert np.allclose(g.weights_to_list(), [0, 1.1, 2.1])
    t = gtn.loads("0\n0 1\n0 0 1\n0 2 1 2 1.1\n2 1 2 3 2.1\n")  # 3, 4 and 5 columns
    assert [t.olabel(i) for i in range(3)] == [1, 2, 3]
    only_nodes = gtn.loads("0\n1\n")
    assert (only_nodes.num_nodes(), only_nodes.num_arcs()) == (2, 0)
    for bad in ("", "1\n", "1 0 0\n0 1", "0\n1 1\n", "0\n1\n0 2\n", "0\n1\n0 1 2 3 4 5\n", "\n\n", "a\n1\n"):
        with pytest.raises(ValueError):  # std::invalid_argument
            gtn.loads(bad)
    with pytest.raises(ValueError):
        gtn.loadtxt(str(tmp_path / "missing.txt"))
    with pytest.raises(ValueError):
        gtn.load(str(tmp_path / "missing.bin"))
    with pytest.raises(ValueError):
        gtn.loadb(b"\x01\x00")  # truncated


# ---------------------------------------------------------------------------------------------
# random sampling


def acyclic(rng, n, extra):
    flags, src, dst, il, ol, w = (np.zeros(n, np.uint8), [], [], [], [], [])
    flags[0] = 1
    flags[-1] = 2
    for i in range(1, n):
        src.append(i - 1)
        dst.append(i)
    for _ in range(extra):
        s = int(rng.integers(0, n - 1))
        src.append(s)
        dst.append(int(rng.integers(s + 1, n)))
    k = len(src)
    il = rng.integers(0, 3, k)
    ol = rng.integers(0, 3, k)
    w = rng.integers(-3, 4, k)
    return (flags, np.array(src, np.int32), np.array(dst, np.int32), il.astype(np.int32), ol.astype(np.int32),
            w.astype(np.float32))


@pytest.mark.parametrize("seed", range(6))
def test_sample_draws_the_reference_path_under_the_same_srand(gtn, seed):
    """Both libraries draw from the C library's rand() in the same order (rand.cpp:14-47)."""
    rng = np.random.default_rng(600 + seed)
    arrs = random_graph(rng, 6, 14, p_eps=0.1) if seed % 2 else acyclic(rng, 7, 6)
    m = ours_from(gtn, arrs)
    for s, want in enumerate(golden("sample", seed)):
        gtn.srand(1000 + s)
        got = gtn.sample(m, 50)
        assert_same(got, want, "sample seed %d" % s)


def test_sample_properties_and_gradient(gtn):
    rng = np.random.default_rng(7)
    arrs = acyclic(rng, 8, 7)
    g = ours_from(gtn, arrs)
    gtn.srand(3)
    p = gtn.sample(g)
    n = p.num_arcs()
    assert n >= 1 and p.num_nodes() == n + 1 and p.is_start(0) and p.is_accept(n)
    assert [p.src_node(i) for i in range(n)] == list(range(n))
    # every arc of the path is an arc of g; the gradient counts how often each was taken
    gtn.backward(p)
    grad = np.array(g.grad().weights_to_list()).reshape(-1)
    assert grad.sum() == n and set(np.unique(grad)) <= {0.0, 1.0}
    taken = np.nonzero(grad)[0]
    assert sorted(arrs[3][taken].tolist()) == sorted(p.labels_to_list())
    # no start node, no accept node, dead end: the empty graph
    assert gtn.sample(gtn.Graph()).num_nodes() == 0
    d = gtn.Graph()
    d.add_node(True)
    d.add_node()
    d.add_arc(0, 1, 0)
    assert gtn.sample(d).num_nodes() == 0
    d.make_accept(0)  # may stop at once: a single accepting node, or walk into the dead end
    for s in range(8):
        gtn.srand(s)
        r = gtn.sample(d)
        assert (r.num_nodes(), r.num_arcs()) in ((0, 0), (1, 0))


# ---------------------------------------------------------------------------------------------
# general composition (both operands arbitrary: epsilons, cycles, any sortedness) is host graph
# construction here as in the reference (compose.cpp:377-522); the device takes over when one
# operand is a gtn::linearGraph (tests/test_gpu_*.py)


@pytest.mark.parametrize("seed", range(24))
def test_general_compose_matches_reference_structure_and_gradients(gtn, seed):
    rng = np.random.default_rng(700 + seed)
    a = random_graph(rng, int(rng.integers(1, 7)), int(rng.integers(0, 14)), n_labels=3, p_eps=0.2)
    b = random_graph(rng, int(rng.integers(1, 7)), int(rng.integers(0, 14)), n_labels=3, p_eps=0.2)
    intersect = seed % 3 == 0
    if intersect:  # acceptors
        a = (a[0], a[1], a[2], a[3], a[3].copy(), a[5])
        b = (b[0], b[1], b[2], b[3], b[3].copy(), b[5])
    ma, mb = ours_from(gtn, a), ours_from(gtn, b)
    if seed & 1:  # the three matchers: unsorted, singly sorted, doubly sorted (functions.cpp:225-251)
        ma.arc_sort(True)
    if seed & 2:
        mb.arc_sort(False)
    mo = gtn.intersect(ma, mb) if intersect else gtn.compose(ma, mb)
    want = golden("compose", seed)
    assert_same(mo, want["out"], "composed graph: same node and arc numbering as the reference")
    assert (want["grads"] is not None) == bool(mo.num_arcs())
    if mo.num_arcs():
        gtn.backward(mo, seed_like(gtn, mo, rng))
        for m, g in zip((ma, mb), want["grads"]):
            assert np.array_equal(np.array(m.grad().weights_to_list(), np.float32).reshape(-1), np.array(g, np.float32))
