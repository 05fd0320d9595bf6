"""Tiled 2-state kernel: (tip, cherry) subtrees computed inside their parent's op (SRC_SMALL).

Trees with such subtrees beside an internal node, a tip, another such subtree and a cherry (the last is not inlined).
Every partial, including the records of inlined nodes read back from the snapshot, must equal the row-major kernel's
bit for bit; lnL must equal the tiled kernel's without inlining bit for bit, in cache-kept, likelihood-only and
dirty-path evaluations; and the tiled pass must run exactly one op fewer per inlined node.

The arithmetic of the inlined op body shows in lnL and in the partials of the nodes above an inlined subtree.  A record
read back through the snapshot is recomputed on demand by an ordinary op, so its comparison checks the record (its
children and the P copies the op images write), not the inlined body."""
import numpy as np
import pytest

import pruning_oracle as oracle
from test_gpu_parity import _random_problem

pytestmark = pytest.mark.gpu


def _build(shape):
    """Nested pairs of tip ids 1..n -> (tree dict, root, n_taxa) with reference-style node ids."""
    rng = np.random.default_rng(11)
    tips = []

    def collect(s):
        if isinstance(s, tuple):
            collect(s[0]), collect(s[1])
        else:
            tips.append(s)
    collect(shape)
    n_taxa = len(tips)
    tree, nxt = {}, [n_taxa + 1]

    def make(s):
        if not isinstance(s, tuple):
            return s
        a, b = make(s[0]), make(s[1])
        node = nxt[0]
        nxt[0] += 1
        tree[node, a] = float(rng.exponential(0.15))
        tree[node, b] = float(rng.exponential(0.15))
        return node
    root = make(shape)
    return tree, root, n_taxa


# (tip, cherry) beside a tip, beside another (tip, cherry), beside an internal node, beside a cherry; all under
# nodes with two internal children so the walk also pushes
HAND = ((((1, (2, 3)), 4), ((5, (6, 7)), ((8, 9), 10))),
        (((11, (12, 13)), ((14, 15), (16, (17, 18)))), (((19, (20, 21)), (22, 23)), ((24, 25), (26, 27)))))


def _expected_inlined(tree, root, n_taxa):
    """Nodes the planner computes inside their parent (full pass, one range): a non-root (tip, cherry) node whose
    sibling is a tip or an internal node that is not a cherry; one per parent."""
    kids = oracle.children_of(tree)
    N = n_taxa
    cherry = {v for v, (a, b) in kids.items() if a <= N and b <= N and v != root}
    is_op = lambda x: x > N and x not in cherry
    small = {v for v, (a, b) in kids.items() if is_op(v) and v != root and
             ((a <= N and b in cherry) or (b <= N and a in cherry))}
    n = 0
    for v, (a, b) in kids.items():
        if is_op(v) and any(s in small and (o <= N or is_op(o)) for s, o in ((a, b), (b, a))):
            n += 1
    return n


def _engine(monkeypatch, codes, C, amb, tiled, small_recs, tm, ekeys):
    from cybayes_b200.engine import Engine
    monkeypatch.setenv("CYBAYES_S2_TILED", tiled)
    monkeypatch.setenv("CYBAYES_S2T_SMALL_RECS", small_recs)
    eng = Engine(codes, 2, C, amb)
    block = eng.alloc_slots(len(ekeys) * C)
    slot_of = {(k, e): block.base + k * len(ekeys) + i for k in range(C) for i, e in enumerate(ekeys)}
    eng.upload_pmats(np.arange(block.base, block.base + block.n, dtype=np.int32),
                     np.stack([tm[k][e] for k in range(C) for e in ekeys]))
    return eng, block, slot_of


@pytest.mark.parametrize("tree_kind,n_cats,minb,v", [("hand", 4, 3, 2), ("hand", 1, 2, 1), ("random64", 4, 3, 2),
                                                     ("random200", 4, 4, 1), ("random200", 1, 3, 2)])
def test_inlined_small_subtrees_match_row_major(tree_kind, n_cats, minb, v, gpu_backend, monkeypatch):
    from cybayes_b200.likelihood import _Plan
    monkeypatch.setenv("CYBAYES_S2T_MINB", str(minb))
    monkeypatch.setenv("CYBAYES_S2T_V", str(v))
    if tree_kind == "hand":
        tree, root, n_taxa = _build(HAND)
        _, _, _, codes, amb, pi, er, rates = _random_problem(77, n_taxa, 700, 2, n_cats=n_cats)
    else:
        n_taxa = int(tree_kind[len("random"):])
        tree, root, _, codes, amb, pi, er, rates = _random_problem(1002, n_taxa, 900, 2, n_cats=n_cats)
    edges = oracle.edge_order(tree, root, n_taxa)
    C = len(rates)
    tm = [oracle.prob_t("GTR", False, pi, tree, er, r) for r in rates]
    plan = _Plan(edges)
    ekeys = list(tree.keys())
    n_inl = _expected_inlined(tree, root, n_taxa)
    assert n_inl >= (3 if tree_kind == "hand" else 1)
    nodes = plan.nodes.tolist()
    parents = oracle.parent_of(tree)

    def dirty(slot_of, tip, swap):
        """the path from `tip` to the root; with `swap` the tip's edge takes another edge's matrices"""
        path = sorted(oracle.path_to_root(parents, tip, root), key=plan.index.__getitem__)
        other = ekeys[(tip * 7) % len(ekeys)]
        ch = np.array([c for n in path for c in plan.kids[n]], dtype=np.int32)
        ps = np.array([[slot_of[k, other if (swap and c == tip) else (n, c)] for k in range(C)]
                       for n in path for c in plan.kids[n]], dtype=np.int32)
        return np.array(path, dtype=np.int32), ch, ps

    tips = list(range(1, n_taxa + 1, max(1, n_taxa // 9)))
    res = {}
    for name, tiled, recs in (("row", "0", "1"), ("inline", "1", "1"), ("plain", "1", "0")):
        eng, block, slot_of = _engine(monkeypatch, codes, C, amb, tiled, recs, tm, ekeys)
        pslots = np.array([[slot_of[k, e] for k in range(C)] for e in plan.edge_keys], dtype=np.int32)
        lnl, snap = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True, force_walk=True)
        full = eng.last_eval_info()
        parts = {n: eng.read_partial(snap, n, with_scale=True) for n in nodes[:-1]}
        lnl_only, _ = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=False, force_walk=True)
        only = eng.last_eval_info()
        paths = []
        for tip in tips:
            same, s1 = eng.eval(snap, *dirty(slot_of, tip, False), pi, want_snapshot=True)
            changed, s2 = eng.eval(snap, *dirty(slot_of, tip, True), pi, want_snapshot=True)
            changed_only, _ = eng.eval(snap, *dirty(slot_of, tip, True), pi, want_snapshot=False)
            path = dirty(slot_of, tip, True)[0].tolist()
            paths.append((same, changed, changed_only, {n: eng.read_partial(s2, n, with_scale=True) for n in path[:-1]}))
            eng.release_snapshot(s1)
            eng.release_snapshot(s2)
        res[name] = (lnl, lnl_only, full, only, parts, paths)
        eng.release_snapshot(snap)
        eng.close()

    (l_r, lo_r, f_r, o_r, p_r, d_r), (l_i, lo_i, f_i, o_i, p_i, d_i), (l_p, lo_p, f_p, o_p, p_p, d_p) = \
        res["row"], res["inline"], res["plain"]
    # lnL: the same bits as the tiled kernel without inlining, within summation order of the row-major kernel
    assert l_i == l_p and lo_i == lo_p and lo_i == l_i
    assert abs(l_i - l_r) <= 1e-13 * abs(l_r)
    # every stored partial and every record (inlined nodes included) equal to the row-major kernel's, bit for bit
    for n in p_r:
        for got in (p_i[n], p_p[n]):
            assert np.array_equal(got[0], p_r[n][0]) and np.array_equal(got[1], p_r[n][1]), n
    # dirty paths: unchanged matrices reproduce the full pass; changed ones agree across kernels
    for (s_i, c_i, co_i, dp_i), (s_p, c_p, co_p, dp_p), (s_r, c_r, co_r, dp_r) in zip(d_i, d_p, d_r):
        assert s_i == l_i and s_p == l_p
        assert c_i == c_p and co_i == c_i and co_p == c_p
        assert abs(c_i - c_r) <= 1e-13 * abs(c_r)
        for n in dp_r:
            assert np.array_equal(dp_i[n][0], dp_r[n][0]) and np.array_equal(dp_i[n][1], dp_r[n][1]), n
    # one kernel op fewer per inlined node; what is stored and written does not change (a likelihood-only pass stores
    # nothing, so it inlines without small records too)
    assert f_p["ops"] == f_r["ops"] and o_p["ops"] == o_i["ops"]
    assert f_r["ops"] - f_i["ops"] == n_inl and o_r["ops"] - o_i["ops"] == n_inl
    assert f_i["stored"] == f_r["stored"] - f_i["small_records"] and f_i["bytes_written"] <= f_r["bytes_written"]
    assert f_i["small_records"] > 0 and f_i["stack_pops"] <= f_p["stack_pops"]
    if tree_kind == "hand":   # ((5, (6, 7)), ((8, 9), 10)): one of the two subtrees was pushed, now neither is
        assert f_i["stack_pops"] < f_p["stack_pops"]
