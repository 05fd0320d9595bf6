"""GPU parity tests (-m gpu): the CUDA path, called through the reference-facing Python surface
and the C ABI, against (a) golden vectors recorded from the unmodified reference, (b) the NumPy
oracle on seeded random inputs, (c) size-independent properties (dirty path == full pass bit for
bit, level schedule == single-launch walk, batch == one by one, scaled == unscaled).

Tolerances: integer artefacts exact; lnL <= 1e-11 relative for JC / F81 (closed forms, same x),
<= 1e-9 relative for GTR (eigendecomposition vs the reference's Pade expm), as BASELINE.json states
(1e-9 relative in fp64)."""
import io
import os
import random
import runpy
import sys

import numpy as np
import pytest

import golden_io
import pruning_oracle as oracle
from conftest import REPO, load_trace

pytestmark = pytest.mark.gpu

REL_CLOSED, REL_GTR = 1e-11, 1e-9


def _setup_case(case):
    from cybayes_b200 import config
    from cybayes_b200.driver import load_alignment
    load_alignment(golden_io.data_path(case), case["dtype"], case["reader"])
    config.MODEL, config.NORM_BETA = case["model"], case["norm_beta"]
    return config


ALL_CASES = ["binary_F81", "twoStates_F81", "twoStates_JC", "narrow_F81", "narrow_JC", "narrow_GTR", "broad_F81",
             "phon_ringe_JC", "phon_ringe_F81", "phon_ringe_GTR", "ie42_JC", "ie42_GTR", "ielex2016_JC",
             "ielex_multistate_F81", "german_multistate_JC"]


@pytest.mark.parametrize("name", ALL_CASES)
def test_golden_full_and_dirty(name, golden_cases, gpu_backend):
    from cybayes_b200.mcmc_gamma import (adjlist2reverse_nodes_dict, get_edge_transition_mat, get_path2root,
                                         get_prob_t)
    from cybayes_b200.ML_gamma import cache_matML, matML
    case = golden_cases[name]
    config = _setup_case(case)
    rel = REL_GTR if case["model"] == "GTR" else REL_CLOSED
    assert config.ALPHABET == case["alphabet"] and config.TAXA == case["taxa"]
    tree, pi, rates, edges, site_rates = golden_io.case_state(case)
    if rates is None:  # too many exchangeabilities to store: JC does not use them
        rates = np.ones(1)
    tmats = [get_prob_t(pi, tree, rates, r) for r in site_rates]
    args = (config.N_SITES, config.N_TAXA, config.N_CATS)
    lnl, cache = matML(pi, case["root"], config.LEAF_LLMAT, edges, tmats, *args)
    assert abs(lnl - case["lnL"]) <= rel * abs(case["lnL"]), (lnl, case["lnL"])
    # P(t) sample
    for key, mats in case["pmat_sample"].items():
        e = tuple(int(x) for x in key.split(","))
        for k, ref in enumerate(mats):
            got = np.asarray(tmats[k][e])
            if isinstance(ref, dict):
                np.testing.assert_allclose(got[0], ref["row0"], rtol=1e-9 if case["model"] == "GTR" else 0, atol=1e-15 if case["model"] == "GTR" else 0)
                np.testing.assert_allclose(np.diag(got), ref["diag"], rtol=1e-9 if case["model"] == "GTR" else 0, atol=0)
            elif case["model"] == "GTR":
                np.testing.assert_allclose(got, np.array(ref), rtol=1e-9, atol=1e-15)
            else:
                assert np.array_equal(got, np.array(ref)), (key, k)  # bit-identical closed forms
    # cached partials: per node, per category sums over states and sites
    some = sorted(case["partial_sums"], key=int)
    for node in some[:: max(1, len(some) // 6)]:
        if int(node) == case["root"]:
            continue
        part = cache.partial(int(node))
        got = part.sum(axis=(1, 2))
        np.testing.assert_allclose(got, case["partial_sums"][node], rtol=1e-9 if case["model"] == "GTR" else 1e-12)
    if "partials" in case:
        for node, ref in case["partials"].items():
            if int(node) != case["root"]:
                np.testing.assert_allclose(cache.partial(int(node)), np.array(ref), rtol=1e-13, atol=0)
    # dirty-path evaluations recorded from the reference
    parents = adjlist2reverse_nodes_dict(tree)
    for d in case["dirty"]:
        e = tuple(d["edge"])
        saved = [tmats[k][e] for k in range(len(tmats))]
        for k, r in enumerate(site_rates):
            tmats[k][e] = get_edge_transition_mat(pi, rates, d["new_t"] * r)
        path = get_path2root(parents, e[1], case["root"])
        assert path == d["path"]
        l2, c2 = cache_matML(pi, case["root"], config.LEAF_LLMAT, cache, path, edges, tmats, *args)
        assert abs(l2 - d["lnL"]) <= rel * abs(d["lnL"]), (e, l2, d["lnL"])
        for k in range(len(tmats)):
            tmats[k][e] = saved[k]
    # after restoring, the dirty path over the same nodes reproduces the full pass bit for bit
    l3, _ = cache_matML(pi, case["root"], config.LEAF_LLMAT, cache, path, edges, tmats, *args)
    assert l3 == lnl


def _random_problem(seed, n_taxa, n_sites, S, n_cats=4, missing=0.1, poly=0.02, bl_mean=0.1, n_poly=3, code_dtype=None):
    """Seeded tree, codes, ambiguity sets, pi, exchangeabilities and category rates.  Every category count above 1
    gets the distinct discrete-Gamma rates of alpha = 0.7, so a kernel that mixes up categories gives another lnL.
    code_dtype: np.uint16 forces 2-byte codes where 1 byte would do."""
    rng = np.random.default_rng(seed)
    pyr = random.Random(seed)
    # random topology: join two random subtrees until one is left; ids like the reference
    nodes = list(range(1, n_taxa + 1))
    nxt = n_taxa + 1
    tree = {}
    while len(nodes) > 1:
        a = nodes.pop(pyr.randrange(len(nodes)))
        b = nodes.pop(pyr.randrange(len(nodes)))
        tree[nxt, a] = float(rng.exponential(bl_mean))
        tree[nxt, b] = float(rng.exponential(bl_mean))
        nodes.append(nxt)
        nxt += 1
    root = nxt - 1
    edges = oracle.edge_order(tree, root, n_taxa)
    amb = [np.ones(S)]
    if S > 2 and poly > 0:
        for _ in range(n_poly):
            v = np.zeros(S)
            v[rng.choice(S, size=2, replace=False)] = 1.0
            amb.append(v)
    amb = np.array(amb)
    codes = rng.integers(0, S, size=(n_taxa, n_sites))
    codes[rng.random((n_taxa, n_sites)) < missing] = S
    if len(amb) > 1:
        m = rng.random((n_taxa, n_sites)) < poly
        codes[m] = S + rng.integers(1, len(amb), size=int(m.sum()))
    codes = codes.astype(code_dtype or (np.uint8 if S + len(amb) <= 256 else np.uint16))
    pi = rng.dirichlet(np.full(S, 5.0))
    er = rng.dirichlet(np.ones(S * (S - 1) // 2))
    rates = oracle.site_rates(0.7, n_cats) if n_cats > 1 else [1.0]
    return tree, root, edges, codes, amb, pi, er, rates


def _oracle_leaves(codes, S, amb):
    table = np.vstack([np.eye(S), amb])
    return {t + 1: np.ascontiguousarray(table[codes[t].astype(np.int64)].T) for t in range(codes.shape[0])}


@pytest.mark.parametrize("S,n_taxa,n_sites,model", [(2, 2, 70, "F81"), (5, 3, 10, "GTR"), (2, 12, 333, "F81"),
                                                    (2, 40, 1000, "GTR"), (4, 9, 65, "GTR"), (40, 7, 90, "GTR"),
                                                    (6, 17, 200, "F81"), (23, 14, 129, "JC"), (47, 10, 64, "GTR"),
                                                    (64, 8, 100, "GTR"), (130, 6, 40, "F81"),
                                                    # >= 16384 patterns: the register-carried FP64 tensor kernel by default
                                                    (64, 12, 16500, "GTR"), (47, 9, 16400, "F81")])
def test_random_inputs_vs_oracle(S, n_taxa, n_sites, model, gpu_backend):
    """Engine called directly with host P matrices (cb_pmat_upload) and with device-built ones
    (cb_pmat_build): lnL, every cached partial and the batched P builder against the oracle."""
    _check_random_inputs(S, n_taxa, n_sites, model)


@pytest.mark.parametrize("S,n_taxa,n_sites,model", [(64, 8, 100, "GTR"), (47, 10, 64, "GTR"), (40, 7, 90, "GTR"),
                                                    (32, 9, 300, "F81"), (56, 12, 200, "JC"), (48, 6, 129, "GTR"),
                                                    (64, 33, 1000, "F81"), (33, 7, 70, "GTR"), (46, 8, 130, "F81"),
                                                    (61, 6, 100, "JC")])
def test_random_inputs_register_carried_dmma(S, n_taxa, n_sites, model, gpu_backend, monkeypatch):
    """The same checks with the large-alignment FP64 tensor kernel (kernels_dmma_rc.cuh: partial carried in
    mma fragments, P matrices streamed by bulk-async copies) forced onto small inputs: ragged last blocks
    (64 of 128 sites), padded state counts (47), missing cells and ambiguity sets in every tile."""
    monkeypatch.setenv("CYBAYES_DMMA_RC", "1")
    _check_random_inputs(S, n_taxa, n_sites, model)


@pytest.mark.parametrize("S,n_taxa,n_sites,model", [(23, 14, 129, "JC"), (9, 5, 70, "GTR"), (17, 6, 200, "F81"),
                                                    (31, 7, 90, "GTR"), (16, 9, 64, "F81"), (24, 5, 300, "GTR")])
def test_register_carried_dmma_small_state_counts(S, n_taxa, n_sites, model, gpu_backend, monkeypatch):
    """The register-carried kernel compiled for 16 and 24 padded states (9 <= S < 32)."""
    monkeypatch.setenv("CYBAYES_DMMA_RC", "1")
    monkeypatch.setenv("CYBAYES_RC_MIN_STATES", "9")
    _check_random_inputs(S, n_taxa, n_sites, model)


def test_register_carried_dmma_many_ambiguity_sets(gpu_backend, monkeypatch):
    """More ambiguity sets than the spare rows of a staged tip image (8): codes beyond them take the dense path."""
    monkeypatch.setenv("CYBAYES_DMMA_RC", "1")
    _check_random_inputs(64, 9, 200, "GTR", n_poly=13, poly=0.2)


def _check_random_inputs(S, n_taxa, n_sites, model, **problem):
    from cybayes_b200 import _lib
    from cybayes_b200.engine import Engine
    from cybayes_b200.likelihood import _Plan
    from cybayes_b200.subst import gtr_eigensystem
    tree, root, edges, codes, amb, pi, er, rates = _random_problem(1000 + S, n_taxa, n_sites, S, **problem)
    C = len(rates)
    leaves = _oracle_leaves(codes, S, amb)
    beta = oracle.f81_beta(pi)
    if model == "JC":
        pi = np.full(S, 1.0 / S)
        beta = oracle.f81_beta(pi)
    tm = [oracle.prob_t(model, False, pi, tree, er, r, beta=beta) for r in rates]
    want, want_cache = oracle.mat_ml(pi, root, leaves, edges, tm, n_sites, n_taxa, n_cats=C)
    want_scaled = oracle.mat_ml_scaled(pi, root, leaves, edges, tm, n_sites, n_taxa, n_cats=C)
    assert abs(want - want_scaled) <= 1e-13 * abs(want)

    eng = Engine(codes, S, C, amb)
    plan = _Plan(edges)
    ekeys = list(tree.keys())
    n_e = len(ekeys)
    # (a) host matrices uploaded
    block = eng.alloc_slots(n_e * C)
    slot_of = {(k, e): block.base + k * n_e + i for k in range(C) for i, e in enumerate(ekeys)}
    eng.upload_pmats(np.arange(block.base, block.base + n_e * C, dtype=np.int32),
                     np.stack([tm[k][e] for k in range(C) for e in ekeys]))
    pslots = np.array([[slot_of[k, e] for k in range(C)] for e in plan.edge_keys], dtype=np.int32)
    lnl, snap = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True, store_root=True)
    assert abs(lnl - want) <= 1e-12 * abs(want), (lnl, want)
    for node in plan.nodes.tolist():
        got = eng.read_partial(snap, node)
        ref = np.stack([want_cache[k][node] for k in range(C)])
        np.testing.assert_allclose(got, ref, rtol=1e-12, atol=0)
    # the three schedules (levels / depth-first walk, with and without keeping the cache) agree bit for bit
    l_walk, s_walk = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True, force_walk=True)
    l_walk2, _ = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=False, force_walk=True)
    l_lev, _ = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=False, force_levels=True)
    assert l_walk == lnl and l_walk2 == lnl and l_lev == lnl
    # 2-state family: cherries folded into their parents (default) vs run as ordinary ops: same bits
    l_nf, s_nf = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True, no_fold=True)
    assert l_nf == lnl
    for node in plan.nodes.tolist()[:-1]:
        assert np.array_equal(eng.read_partial(s_nf, node), eng.read_partial(snap, node))
    eng.release_snapshot(s_nf)
    # small shards cut the walk into parallel subtrees + a top part (two launches): same bits
    os.environ["CYBAYES_WALK_SPLIT"] = "3"
    try:
        l_split, s_split = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True, force_walk=True)
        l_split2, _ = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=False, force_walk=True)
    finally:
        del os.environ["CYBAYES_WALK_SPLIT"]
    assert l_split == lnl and l_split2 == lnl
    for node in plan.nodes.tolist()[:-1]:
        assert np.array_equal(eng.read_partial(s_split, node), eng.read_partial(snap, node))
    eng.release_snapshot(s_split)
    for node in plan.nodes.tolist()[:-1]:
        assert np.array_equal(eng.read_partial(s_walk, node), eng.read_partial(snap, node))
    eng.release_snapshot(s_walk)
    # asynchronous form: enqueue now (CB_EVAL_NO_SYNC), collect the number later (cb_result_wait)
    _, s_async = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True, sync=False)
    assert eng.wait() == lnl
    eng.release_snapshot(s_async)
    # (b) device-built matrices
    block2 = eng.alloc_slots(n_e * C)
    slots2 = np.arange(block2.base, block2.base + n_e * C, dtype=np.int32)
    d = np.array([tree[e] * rates[k] for k in range(C) for e in ekeys])
    if model == "GTR":
        eng.queue_build(_lib.CB_MODEL_GTR_EIG, pi, 0.0, gtr_eigensystem(pi, er), slots2, d)
    elif model == "F81":
        eng.queue_build(_lib.CB_MODEL_F81, pi, beta, None, slots2, d)
    else:
        eng.queue_build(_lib.CB_MODEL_JC, pi, beta, None, slots2, d)
    built = eng.download_pmats(slots2)
    ref = np.stack([tm[k][e] for k in range(C) for e in ekeys])
    if model == "GTR":
        np.testing.assert_allclose(built, ref, rtol=2e-9, atol=1e-14)
    else:
        np.testing.assert_allclose(built, ref, rtol=1e-15, atol=2.3e-16)  # device exp: <= 1 ulp of x (abs)
        # with x = exp(-beta d) from the host libm the closed forms are bit-identical
        import math
        x = np.array([math.exp(-beta * v) for v in d.tolist()])
        eng.queue_build(_lib.CB_MODEL_F81 if model == "F81" else _lib.CB_MODEL_JC, pi, beta, None, slots2, d, x)
        assert np.array_equal(eng.download_pmats(slots2), ref)
    pslots2 = pslots - block.base + block2.base
    lnl2, _ = eng.eval(None, plan.nodes, plan.children, pslots2, pi, want_snapshot=False)
    assert abs(lnl2 - want) <= (1e-9 if model == "GTR" else 1e-12) * abs(want)
    # (c) dirty paths: chain walk == level schedule == full recompute, bit for bit
    parents = oracle.parent_of(tree)
    for tip in (1, n_taxa // 2, n_taxa):
        path = oracle.path_to_root(parents, tip, root)
        todo = sorted(path, key=plan.index.__getitem__)
        nodes = np.array(todo, dtype=np.int32)
        ch = np.array([c for n in todo for c in plan.kids[n]], dtype=np.int32)
        ps = np.array([[slot_of[k, (n, c)] for k in range(C)] for n in todo for c in plan.kids[n]], dtype=np.int32)
        l_chain, s1 = eng.eval(snap, nodes, ch, ps, pi, want_snapshot=True)
        l_levels, s2 = eng.eval(snap, nodes, ch, ps, pi, want_snapshot=True, force_levels=True)
        l_nosnap, _ = eng.eval(snap, nodes, ch, ps, pi, want_snapshot=False)
        assert l_chain == lnl and l_levels == lnl and l_nosnap == lnl
        for n in todo[:-1]:
            assert np.array_equal(eng.read_partial(s1, n), eng.read_partial(s2, n))
        eng.release_snapshot(s1)
        eng.release_snapshot(s2)
    # (d) batch of candidate paths in one launch == one by one
    cands, offs, nn, cc, pp = [], [0], [], [], []
    for tip in range(1, n_taxa + 1):
        path = sorted(oracle.path_to_root(parents, tip, root), key=plan.index.__getitem__)
        nn += path
        cc += [c for n in path for c in plan.kids[n]]
        # candidate: the tip's edge takes the matrix of another edge (a different likelihood)
        other = ekeys[(tip * 7) % n_e]
        for n in path:
            for c in plan.kids[n]:
                pp.append([slot_of[k, other if c == tip else (n, c)] for k in range(C)])
        offs.append(len(nn))
    nn, cc, pp = np.array(nn, dtype=np.int32), np.array(cc, dtype=np.int32), np.array(pp, dtype=np.int32)
    got = eng.eval_batch(snap, np.array(offs, dtype=np.int32), nn, cc, pp, pi)
    for b in range(n_taxa):
        lo, hi = offs[b], offs[b + 1]
        one, _ = eng.eval(snap, nn[lo:hi], cc[2 * lo:2 * hi], pp[2 * lo:2 * hi], pi, want_snapshot=False)
        assert got[b] == one
    eng.close()


def test_deep_tree_needs_scaling(gpu_backend):
    """A 1300-taxon caterpillar with long branches underflows the reference (lnL = -inf, SURVEY F3);
    the GPU path rescales per site and must match the scaled oracle."""
    from cybayes_b200.engine import Engine
    from cybayes_b200.likelihood import _Plan
    n_taxa, n_sites, S, C = 1300, 130, 2, 4
    rng = np.random.default_rng(7)
    tree, prev, nxt = {}, 1, n_taxa + 1
    for tip in range(2, n_taxa + 1):
        tree[nxt, prev] = float(rng.exponential(0.5))
        tree[nxt, tip] = float(rng.exponential(0.5))
        prev, nxt = nxt, nxt + 1
    root = nxt - 1
    codes = rng.integers(0, 2, size=(n_taxa, n_sites)).astype(np.uint8)
    pi = np.array([0.3, 0.7])
    rates = oracle.site_rates(0.5)
    # iterative edge order (the recursive restatement would hit the recursion limit here)
    kids = oracle.children_of(tree)
    order, stack = [], [root]
    while stack:
        nd = stack.pop()
        x, y = kids[nd]
        order += [(nd, x), (nd, y)]
        if y > n_taxa:
            stack.append(y)
        if x > n_taxa:
            stack.append(x)
    edges = order[::-1]
    tm = [oracle.prob_t("F81", True, pi, tree, None, r) for r in rates]
    leaves = _oracle_leaves(codes, S, np.ones((1, S)))
    unscaled = oracle.mat_ml(pi, root, leaves, edges, tm, n_sites, n_taxa)[0]
    assert unscaled == -np.inf
    want = oracle.mat_ml_scaled(pi, root, leaves, edges, tm, n_sites, n_taxa)
    eng = Engine(codes, S, C)
    plan = _Plan(edges)
    ekeys = list(tree.keys())
    block = eng.alloc_slots(len(ekeys) * C)
    slot_of = {(k, e): block.base + k * len(ekeys) + i for k in range(C) for i, e in enumerate(ekeys)}
    eng.upload_pmats(np.arange(block.base, block.base + block.n, dtype=np.int32),
                     np.stack([tm[k][e] for k in range(C) for e in ekeys]))
    pslots = np.array([[slot_of[k, e] for k in range(C)] for e in plan.edge_keys], dtype=np.int32)
    lnl, snap = eng.eval(None, plan.nodes, plan.children, pslots, pi)
    assert np.isfinite(lnl) and abs(lnl - want) <= 1e-12 * abs(want), (lnl, want)
    # the deepest dirty path (1299 nodes > the single-launch limit) falls back to levels: same bits
    parents = oracle.parent_of(tree)
    path = sorted(oracle.path_to_root(parents, 1, root), key=plan.index.__getitem__)
    nodes = np.array(path, dtype=np.int32)
    ch = np.array([c for n in path for c in plan.kids[n]], dtype=np.int32)
    ps = np.array([[slot_of[k, (n, c)] for k in range(C)] for n in path for c in plan.kids[n]], dtype=np.int32)
    l2, _ = eng.eval(snap, nodes, ch, ps, pi, want_snapshot=False)
    assert l2 == lnl
    short = path[-100:]
    nodes = np.array(short, dtype=np.int32)
    ch = np.array([c for n in short for c in plan.kids[n]], dtype=np.int32)
    ps = np.array([[slot_of[k, (n, c)] for k in range(C)] for n in short for c in plan.kids[n]], dtype=np.int32)
    l3, _ = eng.eval(snap, nodes, ch, ps, pi, want_snapshot=False)
    assert l3 == lnl
    eng.close()


from trace_checks import TRACES, check_outputs, compare_trace as _compare_trace  # noqa: E402


@pytest.mark.parametrize("name,n_gen", TRACES)
def test_driver_trace_matches_reference(name, n_gen, golden_cases, gpu_backend, tmp_path):
    """Identical accept/reject trace for a fixed seed: the restated driver on the CUDA engine vs the
    per-generation output recorded from the unmodified reference driver."""
    from cybayes_b200.driver import run_chain
    case = golden_cases[name]
    rows, meta = load_trace(name)
    rec = []
    res = run_chain(golden_io.data_path(case), case["model"], n_gen, 1, case["dtype"], str(tmp_path / "run"),
                    out=io.StringIO(), fast_spr=False,
                    on_generation=lambda i, cur, prop, p, mv, acc, st: rec.append((i, cur, prop, p, mv, acc)))
    rel = REL_GTR if case["model"] == "GTR" else REL_CLOSED
    _compare_trace(rec, rows[:n_gen], meta, res["initial_lnL"], rel)
    check_outputs(str(tmp_path / "run"), rows[:n_gen], meta, res)


@pytest.mark.parametrize("name,n_gen", TRACES)
def test_native_chain_trace_matches_reference(name, n_gen, golden_cases, gpu_backend, tmp_path):
    """The same traces with the generation loop inside the library (cb_chain_*, csrc/mcmc_native.cuh): proposals, P
    matrices, dirty-path evaluation and the accept test without returning to Python between generations."""
    from cybayes_b200.fastchain import run_chain_native
    case = golden_cases[name]
    rows, meta = load_trace(name)
    rec = []
    res = run_chain_native(golden_io.data_path(case), case["model"], n_gen, 1, case["dtype"], str(tmp_path / "run"),
                           out=io.StringIO(),
                           on_generation=lambda i, cur, prop, p, mv, acc, st: rec.append((i, cur, prop, p, mv, acc)))
    rel = REL_GTR if case["model"] == "GTR" else REL_CLOSED
    _compare_trace(rec, rows[:n_gen], meta, res["initial_lnL"], rel)
    check_outputs(str(tmp_path / "run"), rows[:n_gen], meta, res)


def test_fast_spr_same_trace(golden_cases, gpu_backend, tmp_path):
    """Dirty-path scoring of external SPR proposals gives the same chain as the full passes."""
    from cybayes_b200.driver import run_chain
    case = golden_cases["narrow_F81"]
    rows, meta = load_trace("narrow_F81")
    rec = []
    res = run_chain(golden_io.data_path(case), "F81", 1500, 1, "bin", str(tmp_path / "run"), out=io.StringIO(),
                    fast_spr=True, on_generation=lambda i, cur, prop, p, mv, acc, st: rec.append((i, cur, prop, p, mv, acc)))
    _compare_trace(rec, rows[:1500], meta, res["initial_lnL"], REL_CLOSED)


def test_unmodified_reference_driver_runs_on_the_engine(golden_cases, gpu_backend, tmp_path, monkeypatch, capsys):
    """The reference's own driver script, byte-compiled and unmodified (oracle/_ref), on top of the
    compat modules: same per-generation output as when it ran on the reference's own modules."""
    pyc = os.path.join(REPO, "oracle", "_ref", "mat_mcmc_gamma.code")
    if not os.path.exists(pyc):
        pytest.skip("oracle/_ref/mat_mcmc_gamma.code not built (oracle/build_ref.sh)")
    compat = os.path.join(REPO, "cybayes_b200", "compat")
    monkeypatch.syspath_prepend(compat)
    for m in ("config", "utils", "mcmc_gamma", "ML_gamma", "mcmc", "ML"):
        monkeypatch.delitem(sys.modules, m, raising=False)
    case = golden_cases["narrow_F81"]
    n_gen = 1000
    monkeypatch.setattr(sys, "argv", ["mat_mcmc_gamma.py", "-i", golden_io.data_path(case), "-m", "F81", "-n",
                                      str(n_gen), "-t", "1", "-d", "bin", "-o", str(tmp_path / "ref_run")])
    runpy.run_path(pyc, run_name="__main__")
    out = capsys.readouterr().out
    rows, meta = load_trace("narrow_F81")
    gens = [l.split("\t") for l in out.splitlines() if l.split("\t")[0].isdigit() and len(l.split("\t")) == 6]
    assert len(gens) == n_gen
    for f, g in zip(gens, rows):
        assert f[4] == g["param"] and f[5] == g["move"], (f, g)
        assert abs(float(f[2]) - float(g["proposed_ll"])) <= REL_CLOSED * abs(float(g["proposed_ll"])), (f, g)
        assert f[3] == g["TL"], (f, g)
    for m in ("config", "utils", "mcmc_gamma", "ML_gamma", "mcmc", "ML"):
        sys.modules.pop(m, None)


@pytest.mark.parametrize("name,fname,model,dtype,n_gen", [("ng_binary_F81", "binary.phy", "F81", "bin", 300),
                                                          ("ng_phon_ringe_JC", "phon_ringe.phy", "JC", "multi", 300),
                                                          ("ng_narrow_F81", "narrow.phy", "F81", "bin", 400)])
def test_unmodified_non_gamma_driver_runs_on_the_engine(name, fname, model, dtype, n_gen, gpu_backend, tmp_path,
                                                        monkeypatch, capsys):
    """The reference's single-rate driver mat_mcmc.py, unmodified, on the CUDA engine (n_cats = 1)."""
    from conftest import check_nongamma_trace, run_reference_script
    out = run_reference_script("mat_mcmc", ["-i", os.path.join(REPO, "tests", "golden", "data", fname), "-m", model,
                                            "-n", str(n_gen), "-t", "1", "-d", dtype, "-o", str(tmp_path / "ng")],
                               monkeypatch, capsys)
    check_nongamma_trace(out, name, REL_CLOSED)


@pytest.mark.parametrize("name", ["phon_ringe_F81", "narrow_F81", "ielex_multistate_F81"])
def test_batched_nni_scoring(name, golden_cases, gpu_backend):
    """SURVEY 8d/C3: every NNI neighbour of the start tree scored against one cache in ONE launch
    (ML_gamma.score_proposals): bit-identical to cache_matML per candidate, and equal to the oracle's
    dirty-path likelihood (ML_gamma.pyx:83-118) for a sample of candidates."""
    from cybayes_b200.mcmc_gamma import (adjlist2nodes_dict, adjlist2reverse_nodes_dict, get_path2root, get_prob_t,
                                         postorder)
    from cybayes_b200.ML_gamma import cache_matML, matML, score_proposals
    case = golden_cases[name]
    config = _setup_case(case)
    tree, pi, rates, edges, site_rates = golden_io.case_state(case)
    if rates is None:
        rates = np.ones(1)
    tmats = [get_prob_t(pi, tree, rates, r) for r in site_rates]
    args = (config.N_SITES, config.N_TAXA, config.N_CATS)
    root, N = case["root"], case["n_taxa"]
    lnl, cache = matML(pi, root, config.LEAF_LLMAT, edges, tmats, *args)
    kids = adjlist2nodes_dict(tree)
    proposals, trees = [], []
    for (a, b) in list(tree):
        if b <= N:
            continue
        src = kids[a][1] if kids[a][0] == b else kids[a][0]
        for tgt in kids[b]:
            t2 = dict(tree)
            sbl, tbl = t2.pop((a, src)), t2.pop((b, tgt))
            t2[a, tgt], t2[b, src] = tbl, sbl
            tm = []
            for k in range(config.N_CATS):
                tk = tmats[k].copy()
                tk[a, tgt], tk[b, src] = tk[b, tgt], tk[a, src]
                tm.append(tk)
            order = postorder(adjlist2nodes_dict(t2), root)[::-1]
            dirty = [b] + get_path2root(adjlist2reverse_nodes_dict(t2), b, root)
            proposals.append((dirty, order, tm))
            trees.append(t2)
    assert len(proposals) == 2 * (N - 2)
    batch = score_proposals(pi, root, config.LEAF_LLMAT, cache, proposals)
    single = [cache_matML(pi, root, config.LEAF_LLMAT, cache, d, o, tm, *args)[0] for d, o, tm in proposals]
    assert batch.tolist() == [float(x) for x in single]
    assert len(set(batch.tolist())) > N // 2            # the candidates really differ
    # oracle: full likelihood of the rearranged tree (same branch lengths moved with the subtrees)
    _, _, _, _, ll, _, n_sites = oracle.read_phylip(golden_io.data_path(case), case["reader"])
    for idx in range(0, len(proposals), max(1, len(proposals) // 5)):
        t2 = trees[idx]
        tm_o = [oracle.prob_t(case["model"], case["dtype"] == "bin", pi, t2, rates, r, beta=case["norm_beta"])
                for r in site_rates]
        want = oracle.mat_ml(pi, root, ll, proposals[idx][1], tm_o, n_sites, N)[0]
        assert abs(batch[idx] - want) <= 1e-11 * abs(want), (idx, batch[idx], want)


def _c1_golden():
    import json
    base = os.path.join(REPO, "tests", "golden", "traces", "c1_narrow_F81_100k")
    meta = json.load(open(base + ".json"))
    z = np.load(base + ".npz")
    log = open(base + ".log").read().splitlines()
    return meta, z["move"], np.unpackbits(z["accepted"])[:len(z["move"])].astype(bool), z["proposed_ll_every_100"], log


@pytest.mark.parametrize("runner", ["driver", "native"])
def test_c1_at_its_stated_length(runner, golden_cases, gpu_backend, tmp_path):
    """Config C1 as the README runs it (README.md:46): narrow.phy, F81, -n 100000 -t 1000, seed 1234.  The restated
    driver on the CUDA engine must take the recorded move and make the recorded accept/reject decision in every one
    of the 100 000 generations (recorded from the unmodified reference, tests/golden/make_golden.py --c1-100k); on a
    mismatch the first divergent generation and the margin |ll_ratio - log u| of its acceptance test are reported
    (SURVEY section 7 (v): a rounding-level flip has a margin <~ 1e-9 * |lnL|)."""
    if runner == "driver":
        from cybayes_b200.driver import run_chain
    else:   # the same chain with the generation loop inside the library
        from cybayes_b200.fastchain import run_chain_native as run_chain
    meta, move, accepted, sampled, log = _c1_golden()
    names = meta["moves"]
    n_gen = len(move)
    got_move = np.empty(n_gen, dtype=np.uint8)
    got_acc = np.empty(n_gen, dtype=bool)
    got_ll = np.empty(n_gen)
    margin = np.empty(n_gen)
    diag = {}

    def rec(i, cur, prop, p, mv, acc, st):
        got_move[i - 1], got_acc[i - 1], got_ll[i - 1] = names.index(mv), acc, prop
        margin[i - 1] = abs(diag["ll_ratio"] - diag["log_u"])
    res = run_chain(golden_io.data_path(golden_cases["narrow_F81"]), "F81", n_gen, 1000, "bin", str(tmp_path / "c1"),
                    out=io.StringIO(), on_generation=rec, diag=diag)
    bad = np.nonzero((got_move != move) | (got_acc != accepted))[0]
    if bad.size:
        g = int(bad[0])
        pytest.fail(f"first divergent generation {g + 1}: move {names[got_move[g]]} (reference {names[move[g]]}), "
                    f"accepted {bool(got_acc[g])} (reference {bool(accepted[g])}), proposed lnL {got_ll[g]!r}, "
                    f"margin |ll_ratio - log u| = {margin[g]:.3e}")
    np.testing.assert_allclose(got_ll[99::100], sampled, rtol=REL_CLOSED, atol=0)
    # the .log of the README command: tree length and alpha exact strings, lnL to 1e-11; final tree and counters exact
    rows = open(str(tmp_path / "c1.log")).read().splitlines()
    assert len(rows) == len(log) and rows[0] == log[0]
    for r, g in zip(rows[1:], log[1:]):
        r, g = r.split("\t"), g.split("\t")
        assert (r[0], r[2], r[3]) == (g[0], g[2], g[3]), (r, g)
        assert abs(float(r[1]) - float(g[1])) <= REL_CLOSED * abs(float(g[1])), (r, g)
    trees = open(str(tmp_path / "c1.trees")).read()
    assert trees.strip().splitlines()[-1].split("\t")[1] == meta["last_tree"]
    import hashlib
    assert hashlib.sha256(trees.encode()).hexdigest() == meta["trees_sha256"]
    counters = sorted(f"({str(k[0])!r}, {k[1]!r}) {res['accepts'].get(k, 0)} {v}" for k, v in res["moves"].items())
    assert counters == sorted(c.replace("np.str_(", "").replace("'),", "',", 1) for c in meta["counters"])
    print(f"C1 100k ({runner}): {res['gens_per_sec']:.0f} generations/s; smallest acceptance margin over the run "
          f"{margin.min():.3e} at generation {int(margin.argmin()) + 1}")


def test_c1_at_its_stated_length_unmodified_script(gpu_backend, tmp_path, monkeypatch, capsys):
    """The same README command through the reference's own, unmodified driver script on the compat modules: its
    .log (TL, alpha exact; lnL 1e-11), its .trees (byte-exact, by digest) and its counters equal the recorded run."""
    import hashlib
    from conftest import run_reference_script
    meta, _, _, _, log = _c1_golden()
    out = run_reference_script("mat_mcmc_gamma", ["-i", os.path.join(REPO, "tests", "golden", "data", "narrow.phy"),
                                                  "-m", "F81", "-n", "100000", "-t", "1000", "-d", "bin", "-o",
                                                  str(tmp_path / "c1ref")], monkeypatch, capsys)
    rows = open(str(tmp_path / "c1ref.log")).read().splitlines()
    assert len(rows) == len(log)
    for r, g in zip(rows[1:], log[1:]):
        r, g = r.split("\t"), g.split("\t")
        assert (r[0], r[2], r[3]) == (g[0], g[2], g[3]), (r, g)
        assert abs(float(r[1]) - float(g[1])) <= REL_CLOSED * abs(float(g[1])), (r, g)
    assert hashlib.sha256(open(str(tmp_path / "c1ref.trees")).read().encode()).hexdigest() == meta["trees_sha256"]
    counters = [l for l in out.splitlines() if l.startswith("(np.str_(") or l.startswith("('")]
    assert sorted(counters) == sorted(meta["counters"])


@pytest.mark.parametrize("n_taxa,n_sites,model,slots,n_cats,minb,bulk,v",
                         [(2, 70, "F81", 3, 4, 2, 0, 2), (12, 333, "F81", 3, 4, 3, 0, 1), (40, 1000, "GTR", 1, 4, 2, 1, 1),
                          (64, 3000, "GTR", 0, 4, 3, 0, 1), (33, 257, "F81", 2, 4, 2, 0, 2), (200, 640, "GTR", 4, 4, 2, 0, 2),
                          (200, 640, "GTR", 3, 4, 3, 1, 1), (25, 500, "F81", 3, 1, 2, 0, 2), (90, 2100, "GTR", 2, 1, 3, 1, 1),
                          (64, 3000, "GTR", 1, 4, 2, 1, 2), (150, 900, "F81", 4, 4, 2, 0, 1), (120, 1500, "GTR", 2, 4, 4, 0, 1),
                          (120, 1500, "F81", 3, 4, 3, 0, 2), (30, 400, "GTR", 2, 1, 4, 0, 1)])
def test_tiled_two_state_kernel_small_inputs(n_taxa, n_sites, model, slots, n_cats, minb, bulk, v, gpu_backend, monkeypatch):
    """The large-alignment 2-state kernel (kernels_s2t.cuh: tile-interleaved partials, shared-memory stack, op images,
    cp.async code ring) forced onto small inputs: ragged last blocks, 0-4 stack slots (spills through global memory),
    both occupancy variants, plain and bulk-async stores, every schedule, dirty paths and batches -- and bit-identical
    partials to the row-major kernel."""
    monkeypatch.setenv("CYBAYES_S2T_MINB", str(minb))
    monkeypatch.setenv("CYBAYES_S2T_BULK", str(bulk))
    monkeypatch.setenv("CYBAYES_S2T_V", str(v))     # tiles per warp
    from cybayes_b200.engine import Engine
    from cybayes_b200.likelihood import _Plan
    monkeypatch.setenv("CYBAYES_S2_TILED", "1")
    monkeypatch.setenv("CYBAYES_S2T_SLOTS", str(slots))
    _check_random_inputs(2, n_taxa, n_sites, model, n_cats=n_cats)
    # same inputs through both kernels: every stored partial equal bit for bit, lnL to summation order
    tree, root, edges, codes, amb, pi, er, rates = _random_problem(1002, n_taxa, n_sites, 2, n_cats=n_cats)
    C = len(rates)
    tm = [oracle.prob_t(model, model == "F81", pi, tree, er, r) for r in rates]
    plan = _Plan(edges)
    ekeys = list(tree.keys())
    res = []
    for tiled in ("1", "0"):
        monkeypatch.setenv("CYBAYES_S2_TILED", tiled)
        eng = Engine(codes, 2, C, amb)
        block = eng.alloc_slots(len(ekeys) * C)
        slot_of = {(k, e): block.base + k * len(ekeys) + i for k in range(C) for i, e in enumerate(ekeys)}
        eng.upload_pmats(np.arange(block.base, block.base + block.n, dtype=np.int32),
                         np.stack([tm[k][e] for k in range(C) for e in ekeys]))
        pslots = np.array([[slot_of[k, e] for k in range(C)] for e in plan.edge_keys], dtype=np.int32)
        lnl, snap = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True, force_walk=True)
        parts = {n: eng.read_partial(snap, n, with_scale=True) for n in plan.nodes.tolist()[:-1]}
        info = eng.last_eval_info()
        res.append((lnl, parts, info))
        eng.close()
    (l1, p1, i1), (l0, p0, i0) = res
    assert abs(l1 - l0) <= 1e-13 * abs(l0)
    for n in p1:
        assert np.array_equal(p1[n][0], p0[n][0]) and np.array_equal(p1[n][1], p0[n][1]), n
    # the tiled kernel keeps small subtrees (children: tips / cherries) as records instead of stored partials
    assert i1["stored"] + i1["small_records"] == i0["stored"] and i0["small_records"] == 0
    assert i1["bytes_written"] <= i0["bytes_written"]
    if slots > 0 and n_taxa > 8:
        assert i1["stack_pops"] > 0 and i1["read_back"] <= i0["read_back"] and i1["small_records"] > 0


@pytest.mark.parametrize("name", ["narrow_F81", "ielex_multistate_F81", "phon_ringe_GTR"])
def test_batched_spr_scoring(name, golden_cases, gpu_backend):
    """External-SPR candidates (mcmc_gamma.pyx:136-185; the reference scores each with a full pass,
    mat_mcmc_gamma.py:167-169) scored as ONE batch against one cache: every candidate is the two dirty paths that
    merge at the regraft point.  Bit-identical to cache_matML per candidate; equal to the oracle's full likelihood of
    the rearranged tree."""
    from cybayes_b200.driver import _spr_dirty_nodes, spr_tables
    from cybayes_b200.mcmc_gamma import adjlist2reverse_nodes_dict, externalSPR, get_prob_t
    from cybayes_b200.ML_gamma import cache_matML, matML, score_proposals
    case = golden_cases[name]
    config = _setup_case(case)
    tree, pi, rates, edges, site_rates = golden_io.case_state(case)
    if rates is None:
        rates = np.ones(1)
    tmats = [get_prob_t(pi, tree, rates, r) for r in site_rates]
    args = (config.N_SITES, config.N_TAXA, config.N_CATS)
    root, N = case["root"], case["n_taxa"]
    lnl, cache = matML(pi, root, config.LEAF_LLMAT, edges, tmats, *args)
    parent_of = adjlist2reverse_nodes_dict(tree)
    random.seed(4242)
    proposals, trees = [], []
    while len(proposals) < 24:
        t2, order, hr = externalSPR(dict(tree), root)
        if hr == 0.0:
            continue                       # the move was a no-op
        dirty = sorted(_spr_dirty_nodes(parent_of, t2, root))
        proposals.append((dirty, order, spr_tables(tmats, t2, pi, rates, site_rates)))
        trees.append(t2)
    batch = score_proposals(pi, root, config.LEAF_LLMAT, cache, proposals)
    single = [cache_matML(pi, root, config.LEAF_LLMAT, cache, d, o, tm, *args)[0] for d, o, tm in proposals]
    assert batch.tolist() == [float(x) for x in single]
    assert len(set(batch.tolist())) > 12
    _, _, _, _, ll, _, n_sites = oracle.read_phylip(golden_io.data_path(case), case["reader"])
    rel = REL_GTR if case["model"] == "GTR" else REL_CLOSED
    for idx in range(0, len(proposals), 4):
        tm_o = [oracle.prob_t(case["model"], case["dtype"] == "bin", pi, trees[idx], rates, r, beta=case["norm_beta"])
                for r in site_rates]
        want = oracle.mat_ml(pi, root, ll, proposals[idx][1], tm_o, n_sites, N)[0]
        assert abs(batch[idx] - want) <= rel * abs(want), (idx, batch[idx], want)


def test_cache_that_does_not_fit_is_lazy_and_fails_cleanly(gpu_backend, monkeypatch):
    """SURVEY 7 / C5 on one GPU: when the partial cache of a full evaluation cannot fit the device, matML evaluates the
    likelihood without keeping partials and hands back a lazy cache; using that cache then fails with a clear
    out-of-memory error instead of a raw cudaMalloc failure.  Reached here with a per-context memory cap."""
    from cybayes_b200 import config
    from cybayes_b200._lib import CyBayesB200Error
    from cybayes_b200.alignment import LeafMatrices
    from cybayes_b200.likelihood import LazyPartialCache
    from cybayes_b200.ML_gamma import cache_matML, matML
    from cybayes_b200.mcmc_gamma import get_prob_t
    from cybayes_b200.synthetic import SyntheticAlignment
    N, P = 64, 81920     # >= 75 776 patterns: the tiled kernel, whose walk keeps read-backs on chip
    aln = SyntheticAlignment(N, P, 2, 77, block_sites=2048)
    codes = aln.codes(0, P)
    monkeypatch.setattr(gpu_backend, "COMPRESS_MAX_SITES", 0)
    monkeypatch.setattr(gpu_backend, "CACHE_CHECK_MIN_BYTES", 0)
    config.N_TAXA, config.N_CHARS, config.N_SITES, config.MODEL, config.IN_DTYPE, config.N_CATS = N, 2, P, "GTR", "bin", 4
    edges = aln.edge_order()

    def evaluate():
        leaves = LeafMatrices(codes, 2, np.ones((1, 2)))
        config.LEAF_LLMAT = leaves
        tabs = [get_prob_t(aln.pi, aln.tree, aln.er, r) for r in aln.rates]
        return leaves, tabs, matML(aln.pi, aln.root, leaves, edges, tabs, P, N, 4)
    _, _, (want, cache) = evaluate()
    assert not isinstance(cache, LazyPartialCache)
    del cache
    gpu_backend.reset_engines()
    # one partial buffer is 81920 * 68 B = 5.6 MB, the full cache up to 62 of them: cap the context at 64 MB
    monkeypatch.setenv("CYBAYES_MAX_DEVICE_BYTES", str(64 << 20))
    leaves, tabs, (lnl, cache) = evaluate()
    assert lnl == want
    assert isinstance(cache, LazyPartialCache)
    parents = oracle.parent_of(aln.tree)
    path = oracle.path_to_root(parents, 5, aln.root)
    with pytest.raises(CyBayesB200Error, match="out of device memory.*shard the patterns"):
        cache_matML(aln.pi, aln.root, leaves, cache, path, edges, tabs, P, N, 4)
    # the context survives the failure (everything the failed evaluation had acquired went back to the pool)
    l2, c2 = matML(aln.pi, aln.root, leaves, edges, tabs, P, N, 4)
    assert l2 == want and isinstance(c2, LazyPartialCache)


@pytest.mark.parametrize("n_taxa,n_sites,n_states", [(64, 300000, 2), (7, 1000, 2), (40, 70000, 23)])
def test_gpu_pattern_compression_equals_the_host_route(n_taxa, n_sites, n_states, gpu_backend):
    """cb_compress_patterns (column hashes on the GPU, grouped on the host, verified column by column on the GPU)
    returns exactly what alignment.compress_patterns returns: same unique columns in order of first appearance, same
    multiplicities, same site -> pattern map (integer artefacts: bit-exact)."""
    from cybayes_b200.alignment import compress_patterns, compress_patterns_gpu
    rng = np.random.default_rng(n_sites)
    base = rng.integers(0, n_states + 1, size=(n_taxa, max(50, n_sites // 40))).astype(np.uint8)   # many repeated columns
    codes = np.ascontiguousarray(base[:, rng.integers(0, base.shape[1], size=n_sites)])
    flip = rng.random(n_sites) < 0.3                                                             # and many singletons
    codes[rng.integers(0, n_taxa, size=int(flip.sum())), np.nonzero(flip)[0]] ^= 1
    p0, w0, m0 = compress_patterns(codes)
    p1, w1, m1 = compress_patterns_gpu(codes)
    assert p0.shape == p1.shape and np.array_equal(p0, p1)
    assert np.array_equal(w0, w1) and np.array_equal(m0, m1)
    assert w1.sum() == n_sites and np.array_equal(p1[:, m1], codes)


def test_long_alignment_is_compressed_on_the_gpu(gpu_backend, monkeypatch):
    """An alignment above the host limit goes through the GPU route inside engine_for; lnL equals the uncompressed
    evaluation to summation order."""
    from cybayes_b200 import config
    from cybayes_b200.alignment import LeafMatrices
    from cybayes_b200.likelihood import engine_for
    from cybayes_b200.ML_gamma import matML
    from cybayes_b200.mcmc_gamma import get_prob_t
    from cybayes_b200.synthetic import SyntheticAlignment
    N, P = 32, 40960
    aln = SyntheticAlignment(N, P, 2, 5, block_sites=2048)
    codes = aln.codes(0, P)
    config.N_TAXA, config.N_CHARS, config.N_SITES, config.MODEL, config.IN_DTYPE, config.N_CATS = N, 2, P, "GTR", "bin", 4
    out = []
    for limit in (0, 1000):     # 0: no compression; 1000: above the host limit -> GPU route
        gpu_backend.reset_engines()
        monkeypatch.setattr(gpu_backend, "COMPRESS_MAX_SITES", limit)
        leaves = LeafMatrices(codes, 2, np.ones((1, 2)))
        config.LEAF_LLMAT = leaves
        tabs = [get_prob_t(aln.pi, aln.tree, aln.er, r) for r in aln.rates]
        lnl, cache = matML(aln.pi, aln.root, leaves, aln.edge_order(), tabs, P, N, 4)
        eng, smap = engine_for(leaves, 4)
        out.append((float(lnl), eng.n_patterns, smap is not None))
        part = cache.partial(aln.root - 1) if (aln.root - 1) in cache.nodes() else None
        assert part is None or part.shape == (4, 2, P)      # per-site view, whatever the compression
        del cache
    (l0, n0, m0), (l1, n1, m1) = out
    assert n0 == P and not m0 and n1 < P and m1
    assert abs(l1 - l0) <= 1e-12 * abs(l0)
