"""Regenerate the fixtures of tests/golden from the REAL reference (oracle/_ref/libgtn_ref.so).

Needs the reference compiled by `make -C oracle ref REF=<gtn source tree>`:
    python tests/golden/make_golden.py [reference] [host] [configs]
(all three when none is named).  The fixtures are small and committed; the tests read only them.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po  # noqa: E402
from tests import util  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def ctc_f64(e, tg, blank=0):
    """float64 CTC loss / gradient (alpha-beta over the same lattice), the 'truth' that
    both fp32 implementations are measured against."""
    e = e.astype(np.float64)
    T, C = e.shape
    lab = [blank]
    for t in tg:
        lab += [int(t), blank]
    L = len(lab)
    NEG = -np.inf

    def preds(l):
        p = [l]
        if l > 0:
            p.append(l - 1)
        if l % 2 == 1 and l > 1 and lab[l] != lab[l - 2]:
            p.append(l - 2)
        return p

    a = np.full(L, NEG)
    a[0] = 0.0
    A = [a]
    for t in range(T):
        n = np.full(L, NEG)
        for l in range(L):
            c = [a[p] for p in preds(l)]
            m = max(c)
            if m > NEG:
                n[l] = m + np.log(sum(np.exp(x - m) for x in c)) + e[t, lab[l]]
        a = n
        A.append(a)
    fin = [a[L - 1]] + ([a[L - 2]] if L > 1 else [])
    m = max(fin)
    s = m + np.log(sum(np.exp(x - m) for x in fin))
    b = np.full(L, NEG)
    b[L - 1] = 0.0
    if L > 1:
        b[L - 2] = 0.0
    occ = np.zeros((T, C))
    for t in range(T - 1, -1, -1):
        nb = np.full(L, NEG)
        al = A[t]
        for l in range(L):
            if b[l] == NEG:
                continue
            v = e[t, lab[l]] + b[l]
            for lp in preds(l):
                if al[lp] > NEG:
                    occ[t, lab[l]] += np.exp(al[lp] + v - s)
                nb[lp] = np.logaddexp(nb[lp], v)
        b = nb
    z = 0.0
    sm = np.zeros((T, C))
    for t in range(T):
        mx = e[t].max()
        ls = mx + np.log(np.exp(e[t] - mx).sum())
        z += ls
        sm[t] = np.exp(e[t] - ls)
    return z - s, sm - occ


def reference_golden():
    out = {}
    # BASELINE.json configs[0]
    e, tg = util.bench_inputs(1, 100, 28, 10)
    l, g, _ = po.ref_ctc_batch(e, tg)
    out["c1_loss"], out["c1_grad"] = l, g
    # one utterance of configs[1] + float64 truth
    e, tg = util.bench_inputs(1, 1000, 64, 100)
    l, g, _ = po.ref_ctc_batch(e, tg)
    l64, g64 = ctc_f64(e[0], tg[0])
    out["c2_loss"], out["c2_grad"] = l, g.astype(np.float32)
    out["c2_loss_f64"], out["c2_grad_f64"] = np.float64(l64), g64
    # ASG, 3 utterances sharing transitions (configs[2] shape, small)
    rng = np.random.default_rng(42)
    B, T, C, U = 3, 20, 8, 4
    ea = rng.uniform(-5, 5, (B, T, C)).astype(np.float32)
    tw = rng.uniform(-5, 5, C + C * C).astype(np.float32)
    ta = [rng.integers(0, C, U).astype(np.int32) for _ in range(B)]
    la, ga, tga, _ = po.ref_asg_batch(ea, tw, ta)
    out.update(asg_e=ea, asg_tw=tw, asg_targets=np.stack(ta), asg_loss=la, asg_grad=ga, asg_tgrad=tga)
    # Viterbi over the dense trellis with integer scores: ties everywhere (configs[3] shape, small)
    ev = rng.integers(-3, 4, (4, 30, 6)).astype(np.float32)
    tv = rng.integers(-2, 3, 6 + 36).astype(np.float32)
    pv, sv, _ = po.ref_viterbi_dense_batch(ev, tv)
    out.update(vit_e=ev, vit_tw=tv, vit_paths=pv, vit_scores=sv)
    # CTC forced alignment with integer scores
    tc = [rng.integers(1, 6, 5).astype(np.int32) for _ in range(4)]
    pc, sc, _ = po.ref_viterbi_ctc_batch(ev, tc)
    out.update(fa_targets=np.stack(tc), fa_paths=pc, fa_scores=sc)
    np.savez_compressed(os.path.join(HERE, "reference_golden.npz"), **out)
    err = np.abs(out["c2_grad"][0] - g64)
    print("reference fp32 vs float64 at T=1000: max abs err %.3e, row-sum drift %.3e"
          % (err.max(), np.abs(out["c2_grad"][0].sum(1)).max()))


# ---------------------------------------------------------------------------------------------------------
# reference_host.json: the graph-level tests (tests/test_host_api.py, test_oracle.py, test_gcompose_emulation.py,
# test_gpu_gcompose.py).  Each entry replays the reference's side of one test on the test's own seeded inputs.


def f32list(a):
    """float32 values as the shortest decimals that read back as the same float32."""
    a = np.asarray(a, np.float32).ravel()
    out = [float(str(x)) for x in a]
    assert np.array_equal(np.array(out, np.float32).view(np.int32), a.view(np.int32))
    return out


def rec(arrays):
    """A graph's arrays -> [flags, src, dst, ilabel, olabel, w] (util.graph_arrays reads it back)."""
    return [np.asarray(arrays[k]).tolist() for k in util.GRAPH_KEYS[:5]] + [f32list(arrays["w"])]


def ref_from(arrs, calc_grad=True):
    return po.RefGraph.from_arrays(*arrs, calc_grad=calc_grad)


def ref_seed_like(out, rng):
    """The reference side of test_host_api.seed_like: random deltas, one per arc of `out`."""
    a = out.arrays()
    d = rng.integers(-5, 6, len(a["src"])).astype(np.float32)
    return ref_from((a["flags"], a["src"], a["dst"], a["ilabel"], a["olabel"], d), calc_grad=False)


def host_golden():
    from tests.test_gcompose_emulation import case
    from tests.test_host_api import acyclic, random_graph
    from tests.test_oracle import rand_graph
    out = {k: {} for k in ("concat", "remove", "rational_grads", "equal", "wire", "sample", "compose", "oracle")}

    for seed in range(6):
        rng = np.random.default_rng(100 + seed)
        theirs = [ref_from(random_graph(rng, int(rng.integers(1, 7)), int(rng.integers(0, 12)))) for _ in range(4)]
        gs = []
        for k in range(5):
            gs += [po.ref_concat(theirs[:k]), po.ref_union(theirs[:k])]
        gs.append(po.ref_concat(theirs[:2]))
        for t in theirs:
            gs += [po.ref_closure(t)] + [po.ref_clone(t, p) for p in range(3)]
        out["concat"][str(seed)] = [rec(g.arrays()) for g in gs]

    for seed in range(8):
        rng = np.random.default_rng(200 + seed)
        t = ref_from(random_graph(rng, int(rng.integers(2, 9)), int(rng.integers(1, 20)), p_eps=0.4))
        gs = [po.ref_remove(t), po.ref_remove(t, 1), po.ref_remove(t, -1, 1), po.ref_remove(t, 0, 2)]
        out["remove"][str(seed)] = [rec(g.arrays()) for g in gs]

    for seed in range(4):
        rng = np.random.default_rng(300 + seed)
        graphs = [random_graph(rng, int(rng.integers(1, 6)), int(rng.integers(1, 9))) for _ in range(3)]
        per_op = []
        for op in (po.ref_concat, po.ref_union, lambda gs: po.ref_closure(gs[0])):
            theirs = [ref_from(g, calc_grad=(i != 1)) for i, g in enumerate(graphs)]
            out_t = op(theirs)
            po.ref_backward_with(out_t, ref_seed_like(out_t, rng))
            used = 1 if op not in (po.ref_concat, po.ref_union) else len(theirs)
            per_op.append([None if (i == 1 and used > 1) else f32list(theirs[i].grad().weights())
                           for i in range(used)])
        out["rational_grads"][str(seed)] = per_op

    for seed in range(10):
        rng = np.random.default_rng(400 + seed)
        n = int(rng.integers(1, 8))
        flags, src, dst, il, ol, w = random_graph(rng, n, int(rng.integers(0, 14)), n_labels=2, p_eps=0.1)
        base = (flags, src, dst, il, ol, w)
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
        t0 = ref_from(base)
        out["equal"][str(seed)] = [[po.ref_equal(t0, ref_from(v)), po.ref_isomorphic(t0, ref_from(v))]
                                   for v in variants]

    for seed in range(5):
        rng = np.random.default_rng(500 + seed)
        n_arcs = int(rng.integers(0, 40))
        arrs = random_graph(rng, int(rng.integers(1, 30)), n_arcs, int_weights=(seed % 2 == 0))
        t = ref_from(arrs)
        binary, text = po.ref_serialise(t, 0), po.ref_serialise(t, 1)
        w = {"bin": binary.hex(), "txt": text.decode(), "repr": po.ref_serialise(t, 2).decode(),
             "dot": po.ref_serialise(t, 3).decode("utf-8"), "graph": rec(t.arrays()),
             "from_bin": rec(po.ref_parse(binary, 0).arrays())}
        if arrs[0].any() and (arrs[0] & 2).any():
            w["from_txt"] = rec(po.ref_parse(text, 1).arrays())
        out["wire"][str(seed)] = w

    for seed in range(6):
        rng = np.random.default_rng(600 + seed)
        t = ref_from(random_graph(rng, 6, 14, p_eps=0.1) if seed % 2 else acyclic(rng, 7, 6))
        out["sample"][str(seed)] = [rec(po.ref_sample(t, 1000 + s, 50).arrays()) for s in range(5)]

    for seed in range(24):
        rng = np.random.default_rng(700 + seed)
        a, b, intersect = case(rng, seed, 7, 14, 0.2)
        ta, tb = ref_from(a), ref_from(b)
        if seed & 1:
            ta.arc_sort(True)
        if seed & 2:
            tb.arc_sort(False)
        to = po.ref_op("intersect" if intersect else "compose", ta, tb)
        c = {"out": rec(to.arrays()), "grads": None}
        if to.num_arcs:
            po.ref_backward_with(to, ref_seed_like(to, rng))
            c["grads"] = [f32list(ta.grad().weights()), f32list(tb.grad().weights())]
        out["compose"][str(seed)] = c

    for seed in range(4):
        rng = np.random.default_rng(100 + seed)
        composed = []
        for _ in range(10):
            n1, n2 = int(rng.integers(2, 8)), int(rng.integers(2, 8))
            eps = bool(rng.integers(0, 2))
            r1, r2 = po.RefGraph.from_arrays(*rand_graph(rng, n1, eps)), po.RefGraph.from_arrays(*rand_graph(rng, n2, eps))
            sort_mode = int(rng.integers(0, 4))
            if sort_mode & 1:
                r1.arc_sort(True)
            if sort_mode & 2:
                r2.arc_sort(False)
            composed += [rec(po.ref_op(name, r1, r2).arrays()) for name in ("compose", "intersect")]
        dags = []
        for _ in range(10):
            n = int(rng.integers(2, 30))
            r = po.RefGraph.from_arrays(*util.random_dag(rng, n, int(rng.integers(n, 4 * n)),
                                                         int_weights=bool(rng.integers(0, 2))))
            scores, grads = [], []
            for name in ("forward_score", "viterbi_score"):
                rs = po.ref_op(name, r)
                scores.append(rs.item())
                po.ref_backward(rs)
                grads.append(f32list(r.grad().weights()))
                po.libref().ref_graph_zero_grad(r.h)
            rp = po.ref_op("viterbi_path", r).arrays()
            dags.append({"scores": f32list(scores), "grads": grads, "path_ilabel": rp["ilabel"].tolist(),
                         "path_w": f32list(rp["w"])})
        out["oracle"][str(seed)] = {"compose": composed, "dags": dags}

    with open(os.path.join(HERE, "reference_host.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"), sort_keys=True)
        f.write("\n")


# ---------------------------------------------------------------------------------------------------------
# reference_configs.npz: tests/test_gpu_config_parity.py, the reference at the BASELINE.json configurations.
# A full gradient batch is tens of MB, so per utterance the fixture keeps the reference's exact error against the
# float64 evaluation (max and mean over every element) and the gradient itself on GRAD_SAMPLE positions: the
# GRAD_TOP ones where the reference is furthest from float64, the rest drawn with a fixed seed.

GRAD_SAMPLE, GRAD_TOP = 128, 32


def grad_sample(gr, g64, seed):
    n = gr.shape[0]
    gr, err = gr.reshape(n, -1), np.abs(gr - g64).reshape(n, -1)
    rng = np.random.default_rng(seed)
    idx = np.zeros((n, GRAD_SAMPLE), np.int32)
    for b in range(n):
        top = np.argsort(err[b], kind="stable")[::-1][:GRAD_TOP]
        rest = np.setdiff1d(np.arange(err.shape[1]), top)
        idx[b] = np.sort(np.concatenate([top, rng.choice(rest, GRAD_SAMPLE - GRAD_TOP, replace=False)]))
    return idx, np.take_along_axis(gr, idx, 1).astype(np.float32), err.max(axis=1), err.mean(axis=1)


def configs_golden():
    from oracle import f64
    out = {}
    # configs[1]: the first 64 utterances of bench.py's batch
    n, T, C, U = 64, 1000, 64, 100
    e, tg = util.bench_inputs(n, T, C, U)
    lr, gr, _ = po.ref_ctc_batch(e, tg)
    g64 = np.stack([f64.ctc_f64(e[b], tg[b])[1] for b in range(n)])
    out["ctc_loss"] = lr
    out["ctc_grad_idx"], out["ctc_grad"], out["ctc_grad_err_max"], out["ctc_grad_err_mean"] = grad_sample(gr, g64, 1)
    # configs[2]: 16 utterances sharing one transitions graph
    n, T, C, U = 16, 500, 64, 50
    rng = np.random.default_rng(41)
    e = rng.uniform(-5, 5, (n, T, C)).astype(np.float32)
    tw = rng.uniform(-5, 5, C + C * C).astype(np.float32)
    tg = [rng.integers(0, C, U).astype(np.int32) for _ in range(n)]
    lr, gr, tgr, _ = po.ref_asg_batch(e, tw, tg)
    g64 = np.stack([f64.asg_f64(e[b], tw, tg[b])[1] for b in range(n)])
    out["asg_loss"], out["asg_tgrad"] = lr, tgr
    out["asg_grad_idx"], out["asg_grad"], out["asg_grad_err_max"], _ = grad_sample(gr, g64, 2)
    # configs[3]: dense Viterbi, one integer-valued utterance, then integer-valued transitions
    n, T, C = 3, 2000, 128
    rng = np.random.default_rng(99)
    e = rng.uniform(-5, 5, (n, T, C)).astype(np.float32)
    e[2] = np.round(e[2])
    tws = (rng.uniform(-5, 5, C + C * C).astype(np.float32), np.round(rng.uniform(-3, 3, C + C * C)).astype(np.float32))
    res = [po.ref_viterbi_dense_batch(e, tw) for tw in tws]
    out["vit_paths"] = np.stack([r[0] for r in res])
    out["vit_scores"] = np.stack([r[1] for r in res])
    # configs[3]: CTC forced alignment, two integer-valued utterances
    n, T, C, U = 8, 2000, 128, 200
    e, tg = util.bench_inputs(n, T, C, U, seed=777)
    e[6:] = np.round(e[6:])
    pr, sr, _ = po.ref_viterbi_ctc_batch(e, tg)
    out["fa_paths"], out["fa_scores"] = pr, sr
    np.savez_compressed(os.path.join(HERE, "reference_configs.npz"), **out)


def main():
    assert po.have_ref(), "build oracle/_ref first: make -C oracle ref REF=<gtn source tree>"
    todo = sys.argv[1:] or ["reference", "host", "configs"]
    for name in todo:
        {"reference": reference_golden, "host": host_golden, "configs": configs_golden}[name]()


if __name__ == "__main__":
    main()
