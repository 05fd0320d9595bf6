"""Per-site log-likelihoods and rate-category posteriors (cb_eval_sites, cb_chain_site_lnl, Engine.eval_sites,
likelihood.site_log_likelihoods, NativeChain.site_lnl, the drivers' --site-lnl).

CPU: the host logic on an oracle-backed fake engine -- per-column expansion, the three cache routes, the compressed and
uncompressed alignments, and both drivers writing .sitelnl without touching .log, .trees or stdout.
GPU: every compiled pruning kernel's root epilogue against the scaled oracle, bit-identity across schedules, shard
slices, the C4 kernel at its own shape, a tree that underflows the reference, and the native chain."""
import io
import os

import numpy as np
import pytest

import golden_io
import pruning_oracle as oracle
from conftest import REPO, load_trace
from fake_engine import FakeEngine

NARROW = os.path.join(REPO, "tests", "golden", "data", "narrow.phy")


class SiteFakeEngine(FakeEngine):
    """FakeEngine with eval_sites: the oracle's unscaled pass, root terms summed in the kernels' order.  Products go
    through einsum's own loops instead of BLAS, so that a column's value does not depend on how many columns the
    array has (as on the GPU, where every site is computed on its own): compressed and uncompressed alignments can
    then be compared bit for bit."""

    def _run(self, snapshot, nodes, children, pslots, pi):
        base = self.snaps[snapshot] if snapshot is not None else {}
        new = {}
        C = self.n_cats
        for i, node in enumerate(np.asarray(nodes).tolist()):
            acc = None
            for kx in range(2):
                ch = int(children[2 * i + kx])
                src = [self.leaves[ch]] * C if ch <= self.n_taxa else (new[ch] if ch in new else base[ch])
                v = np.stack([np.einsum("ij,jp->ip", self.pm[int(pslots[2 * i + kx, c])], src[c]) for c in range(C)])
                acc = v if acc is None else acc * v
            new[node] = acc
        ll = np.zeros(self.n_patterns)
        for t in self._terms(pi, new[int(nodes[-1])]):
            ll += t
        with np.errstate(divide="ignore"):
            lnl = float(np.sum(self.weights * np.log(ll)))
        return lnl, base, new

    def _terms(self, pi, root):
        return [np.einsum("i,ip->p", pi, root[c]) / (self.n_cats * 1.0) for c in range(self.n_cats)]

    def eval_sites(self, snapshot, nodes, children, pslots, pi, want_snapshot=False, categories=False):
        pi = np.asarray(pi, dtype=float)
        lnl, base, new = self._run(snapshot, nodes, children, pslots, pi)
        terms = self._terms(pi, new[int(nodes[-1])])
        s = np.zeros(self.n_patterns)
        for t in terms:
            s += t
        with np.errstate(divide="ignore"):
            site = np.log(s)
        sid = -1
        if want_snapshot:
            merged = dict(base)
            merged.update(new)
            sid = self._next_snap
            self._next_snap += 1
            self.snaps[sid] = merged
        return lnl, site, (np.array(terms) / s if categories else None), sid


@pytest.fixture
def site_backend(monkeypatch):
    from cybayes_b200 import likelihood
    likelihood.reset_engines()
    likelihood._plan_cache.clear()
    monkeypatch.setattr(likelihood, "_engine_factory", SiteFakeEngine)
    yield SiteFakeEngine
    likelihood.reset_engines()


def _narrow_state(golden_cases):
    from cybayes_b200 import config
    from cybayes_b200.driver import load_alignment
    case = golden_cases["narrow_F81"]
    load_alignment(golden_io.data_path(case), case["dtype"], case["reader"])
    config.MODEL, config.NORM_BETA = case["model"], case["norm_beta"]
    tree, pi, rates, edges, site_rates = golden_io.case_state(case)
    return case, tree, pi, rates, edges, site_rates


def _surface(golden_cases, monkeypatch, lazy=False):
    """site_log_likelihoods on narrow_F81 through no cache, the matML cache (root only) and a lazy cache."""
    from cybayes_b200 import config, likelihood
    from cybayes_b200.mcmc_gamma import get_prob_t
    from cybayes_b200.ML_gamma import matML
    case, tree, pi, rates, edges, site_rates = _narrow_state(golden_cases)
    tmats = [get_prob_t(pi, tree, rates, r) for r in site_rates]
    root = case["root"]
    if lazy:
        monkeypatch.setattr(likelihood, "LAZY_CACHE_MIN_SITES", 0)
    lnl, cache = matML(pi, root, config.LEAF_LLMAT, edges, tmats, config.N_SITES, config.N_TAXA, config.N_CATS)
    out = {"none": likelihood.site_log_likelihoods(pi, root, config.LEAF_LLMAT, edges, tmats, categories=True),
           "cache": likelihood.site_log_likelihoods(pi, root, config.LEAF_LLMAT, edges, tmats, cache=cache,
                                                    categories=True)}
    if lazy:
        assert isinstance(cache, likelihood.LazyPartialCache) and cache._snap is None   # not materialised
    return case, tree, pi, rates, edges, site_rates, lnl, out


def _root_terms(pi, root, edges, tm, kept, leaf):
    """The per-category root terms pi . L_c,p / n_cats of the oracle's scaled pass, rebuilt from the root's two children
    as mat_ml_scaled keeps them (`kept`: node -> (mantissas (C, S, P), exponents)) with the oracle's own products; tips
    come from `leaf(tip)`.  The terms carry the children's per-site exponent, common to all categories, which cancels in
    the posterior terms / sum(terms)."""
    C = len(tm)
    terms = []
    for k in range(C):
        L = None
        for parent, child in edges:
            if parent == root:
                v = tm[k][root, child].dot(kept[child][0][k] if child in kept else leaf(child))
                L = v if L is None else L * v
        terms.append(np.dot(pi, L) / (C * 1.0))
    return np.array(terms)


def _oracle_sites(pi, root, leaves, edges, tm, n_sites, n_taxa):
    """Scaled oracle: (per-site l, per-category root terms)."""
    keep = {c: None for p, c in edges if p == root and c > n_taxa}
    _, per_site = oracle.mat_ml_scaled(pi, root, leaves, edges, tm, n_sites, n_taxa, n_cats=len(tm), site_lnl=True,
                                       keep=keep)
    return per_site, _root_terms(pi, root, edges, tm, keep, leaves.__getitem__)


@pytest.mark.parametrize("lazy", [False, True])
def test_site_log_likelihoods_equal_the_oracle_per_column(lazy, golden_cases, site_backend, monkeypatch):
    case, tree, pi, rates, edges, site_rates, lnl, out = _surface(golden_cases, monkeypatch, lazy)
    _, _, _, _, ll, _, n_sites = oracle.read_phylip(golden_io.data_path(case), case["reader"])
    tm = [oracle.prob_t("F81", True, pi, tree, rates, r, beta=case["norm_beta"]) for r in site_rates]
    per_site, terms = _oracle_sites(pi, case["root"], ll, edges, tm, n_sites, case["n_taxa"])
    q = terms / terms.sum(axis=0)
    for route, (l_r, site, post) in out.items():
        assert site.shape == (n_sites,) and post.shape == (len(site_rates), n_sites), route
        np.testing.assert_allclose(site, per_site, rtol=1e-11, atol=0)
        np.testing.assert_allclose(post, q, rtol=0, atol=1e-12)
        assert abs(site.sum() - lnl) <= 1e-11 * abs(lnl) and l_r == lnl, route
    assert np.array_equal(out["none"][1], out["cache"][1]) and np.array_equal(out["none"][2], out["cache"][2])


def test_compressed_and_uncompressed_routes_agree(golden_cases, site_backend, monkeypatch):
    from cybayes_b200 import likelihood
    _, _, _, _, _, _, _, a = _surface(golden_cases, monkeypatch)
    eng_a = site_backend.instances[-1]
    likelihood.reset_engines()
    monkeypatch.setattr(likelihood, "COMPRESS_MAX_SITES", 0)
    _, _, _, _, _, _, _, b = _surface(golden_cases, monkeypatch)
    eng_b = site_backend.instances[-1]
    assert eng_a.n_patterns < eng_b.n_patterns          # the first engine really held compressed patterns
    for route in a:
        assert np.array_equal(a[route][1], b[route][1]) and np.array_equal(a[route][2], b[route][2]), route


def _read_sitelnl(path):
    lines = open(path).read().splitlines()
    return lines[0].split("\t"), [[float(x) for x in line.split("\t")] for line in lines[1:]]


def _runs_with_and_without(runner, tmp_path, backend, n_gen, thin, **kw):
    from cybayes_b200 import likelihood
    outs = {}
    for tag, flag in (("plain", False), ("sites", True)):
        likelihood.reset_engines()
        buf = io.StringIO()
        runner(NARROW, "F81", n_gen, thin, "bin", str(tmp_path / tag), out=buf, site_lnl=flag, **kw)
        outs[tag] = buf.getvalue()
    for ext in (".log", ".trees"):
        assert open(str(tmp_path / ("plain" + ext)), "rb").read() == open(str(tmp_path / ("sites" + ext)), "rb").read()
    assert outs["plain"] == outs["sites"]
    assert not os.path.exists(str(tmp_path / "plain.sitelnl"))
    head, rows = _read_sitelnl(str(tmp_path / "sites.sitelnl"))
    _, _, _, _, _, _, n_cols = oracle.read_phylip(NARROW, "readBinaryPhy")
    assert head == ["Iter"] + [str(i) for i in range(1, n_cols + 1)]
    log = [line.split("\t") for line in open(str(tmp_path / "sites.log")).read().splitlines()[1:]]
    assert len(rows) == len(log) == n_gen // thin
    for row, lr in zip(rows, log):
        assert len(row) == 1 + n_cols and row[0] == int(lr[0])
        want = float(lr[1])
        assert abs(sum(row[1:]) - want) <= 1e-11 * abs(want), (row[0], sum(row[1:]), want)
    return rows


def test_python_driver_writes_sitelnl_and_nothing_else_changes(site_backend, tmp_path):
    from cybayes_b200.driver import run_chain
    _runs_with_and_without(run_chain, tmp_path, site_backend, 300, 20, fast_spr=True)


def test_native_loop_on_callbacks_writes_sitelnl_and_nothing_else_changes(site_backend, tmp_path):
    from cybayes_b200.fastchain import run_chain_native
    rows = _runs_with_and_without(run_chain_native, tmp_path, site_backend, 300, 20)
    from cybayes_b200.driver import run_chain
    from cybayes_b200 import likelihood
    likelihood.reset_engines()
    run_chain(NARROW, "F81", 300, 20, "bin", str(tmp_path / "py"), out=io.StringIO(), site_lnl=True)
    _, py_rows = _read_sitelnl(str(tmp_path / "py.sitelnl"))
    np.testing.assert_allclose(np.array(rows), np.array(py_rows), rtol=1e-11, atol=0)


def test_chain_site_lnl_needs_an_eval_sites_callback(golden_cases, site_backend, monkeypatch):
    from cybayes_b200 import config, fastchain, likelihood
    from cybayes_b200._lib import CyBayesB200Error
    from cybayes_b200.mcmc_gamma import get_siterates, state_init
    real = fastchain.engine_callbacks
    monkeypatch.setattr(fastchain, "engine_callbacks", lambda eng: real(eng)[:3] + (fastchain._EVAL_SITES_FN(),))
    _narrow_state(golden_cases)
    config.MODEL = "F81"
    state = state_init()
    eng, _ = likelihood.engine_for(config.LEAF_LLMAT, config.N_CATS)
    chain = fastchain.NativeChain(eng, state, get_siterates(state["srates"]), "F81", True)
    with pytest.raises(CyBayesB200Error, match="eval_sites callback"):
        chain.site_lnl()
    chain.close()


def test_site_lnl_is_refused_on_a_sharded_run(monkeypatch, tmp_path, capsys):
    from cybayes_b200.driver import main
    monkeypatch.setenv("CYBAYES_SHARD", "1")
    with pytest.raises(SystemExit):
        main(["-i", NARROW, "-m", "F81", "-n", "10", "-t", "5", "-d", "bin", "-o", str(tmp_path / "x"), "--site-lnl"])
    assert "CYBAYES_SHARD=1" in capsys.readouterr().err
    from cybayes_b200 import likelihood
    with pytest.raises(ValueError, match="CYBAYES_SHARD=1"):
        likelihood.site_log_likelihoods(np.ones(2) / 2, 3, {}, [], [])


# ------------------------------------------------------------------------------------------------------------ GPU
def _engine_problem(case):
    from cybayes_b200.engine import Engine
    from cybayes_b200.likelihood import _Plan
    from test_gpu_parity import _oracle_leaves, _random_problem
    S, C, n_taxa, n_sites = case["S"], case["C"], case["n_taxa"], case["n_sites"]
    tree, root, edges, codes, amb, pi, er, rates = _random_problem(1000 + S, n_taxa, n_sites, S, n_cats=C,
                                                                   code_dtype=case["dtype"])
    beta = oracle.f81_beta(pi)
    if case["model"] == "JC":
        pi = np.full(S, 1.0 / S)
        beta = oracle.f81_beta(pi)
    tm = [oracle.prob_t(case["model"], False, pi, tree, er, r, beta=beta) for r in rates]
    leaves = _oracle_leaves(codes, S, amb)
    eng = Engine(codes, S, C, amb)
    plan = _Plan(edges)
    from large_cases import _engine_inputs
    _, slot_of, pslots = _engine_inputs(eng, plan, tree, tm, C)
    return dict(tree=tree, root=root, edges=edges, codes=codes, amb=amb, pi=pi, tm=tm, leaves=leaves, eng=eng,
                plan=plan, slot_of=slot_of, pslots=pslots, C=C, n_taxa=n_taxa, n_sites=n_sites)


def _check_against_oracle(site, post, lnl, per_site, terms, rel=1e-11):
    assert np.all(np.isfinite(site))
    assert np.all(np.abs(site - per_site) <= rel * np.maximum(1.0, np.abs(per_site))), \
        np.max(np.abs(site - per_site) / np.maximum(1.0, np.abs(per_site)))
    q = terms / terms.sum(axis=0)
    assert np.max(np.abs(post - q)) <= 1e-12, np.max(np.abs(post - q))
    assert np.max(np.abs(post.sum(axis=0) - 1.0)) <= 1e-14
    assert abs(site.sum() - lnl) <= 1e-12 * abs(lnl), (site.sum(), lnl)


from test_kernel_coverage import CASES  # noqa: E402


@pytest.mark.gpu
@pytest.mark.parametrize("cid", list(CASES))
def test_root_epilogue_of_every_kernel(cid, gpu_backend, monkeypatch):
    """Every compiled pruning kernel's root epilogue: l and q against the scaled oracle, lnL equal to cb_eval's, and
    the same bits from every schedule that ends in that epilogue."""
    case = CASES[cid]
    for k, v in case["env"].items():
        monkeypatch.setenv(k, v)
    p = _engine_problem(case)
    eng, plan, pslots, pi, root, C = p["eng"], p["plan"], p["pslots"], p["pi"], p["root"], p["C"]
    per_site, terms = _oracle_sites(pi, root, p["leaves"], p["edges"], p["tm"], p["n_sites"], p["n_taxa"])
    l_eval, _ = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=False)
    lnl, site, post, snap = eng.eval_sites(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True,
                                           categories=True)
    assert lnl == l_eval
    _check_against_oracle(site, post, lnl, per_site, terms)
    runs = {"levels": dict(force_levels=True), "walk": dict(force_walk=True), "no_fold": dict(no_fold=True)}
    for name, kw in runs.items():
        l2, s2, q2, _ = eng.eval_sites(None, plan.nodes, plan.children, pslots, pi, categories=True, **kw)
        assert l2 == lnl and np.array_equal(s2, site) and np.array_equal(q2, post), name
    kids = plan.kids
    ps_root = np.array([[p["slot_of"][k, (root, c)] for k in range(C)] for c in kids[root]], dtype=np.int32)
    l3, s3, q3, _ = eng.eval_sites(snap, np.array([root], dtype=np.int32), np.array(kids[root], dtype=np.int32),
                                   ps_root, pi, categories=True)
    assert l3 == lnl and np.array_equal(s3, site) and np.array_equal(q3, post), "root only"
    path = sorted(oracle.path_to_root(oracle.parent_of(p["tree"]), 1, root), key=plan.index.__getitem__)
    ch = np.array([c for n in path for c in kids[n]], dtype=np.int32)
    ps = np.array([[p["slot_of"][k, (n, c)] for k in range(C)] for n in path for c in kids[n]], dtype=np.int32)
    l4, s4, q4, _ = eng.eval_sites(snap, np.array(path, dtype=np.int32), ch, ps, pi, categories=True)
    assert l4 == lnl and np.array_equal(s4, site) and np.array_equal(q4, post), "dirty path"
    l5, s5, q5, _ = eng.eval_sites(None, plan.nodes, plan.children, pslots, pi)
    assert l5 == lnl and np.array_equal(s5, site) and q5 is None
    if cid == "s2_c4":   # the flag check sits before any launch: once is enough
        import ctypes
        from cybayes_b200._lib import CB_EVAL_NO_SYNC, CyBayesB200Error, c_f64p, c_i32p, check
        out, l_out, snap_out = np.empty(eng.n_patterns), np.zeros(1), ctypes.c_int()
        pi_c = np.ascontiguousarray(pi, dtype=np.float64)
        with pytest.raises(CyBayesB200Error, match="CB_EVAL_NO_SYNC"):
            check(eng._lib.cb_eval_sites(eng._ctx, -1, plan.nodes.size, plan.nodes.ctypes.data_as(c_i32p),
                                         plan.children.ctypes.data_as(c_i32p), pslots.ctypes.data_as(c_i32p),
                                         pi_c.ctypes.data_as(c_f64p), CB_EVAL_NO_SYNC, ctypes.byref(snap_out),
                                         l_out.ctypes.data_as(c_f64p), out.ctypes.data_as(c_f64p), None))
    eng.release_snapshot(snap)
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cid", ["s2_c4", "general_s7"])
def test_shard_slices_concatenate_to_the_whole(cid, gpu_backend):
    """Two contexts over the two halves of an alignment (cut at a multiple of 64), as two ranks of a site-sharded run
    hold them: their slices, concatenated, are the whole alignment's l and q bit for bit."""
    from cybayes_b200.engine import Engine
    p = _engine_problem(CASES[cid])
    plan, pi, C, codes, amb = p["plan"], p["pi"], p["C"], p["codes"], p["amb"]
    _, site, post, _ = p["eng"].eval_sites(None, plan.nodes, plan.children, p["pslots"], pi, categories=True)
    p["eng"].close()
    cut = 192
    parts = []
    for lo, hi in ((0, cut), (cut, codes.shape[1])):
        eng = Engine(np.ascontiguousarray(codes[:, lo:hi]), len(pi), C, amb)
        from large_cases import _engine_inputs
        _, _, ps = _engine_inputs(eng, plan, p["tree"], p["tm"], C)
        parts.append(eng.eval_sites(None, plan.nodes, plan.children, ps, pi, categories=True)[1:3])
        eng.close()
    assert np.array_equal(np.concatenate([a for a, _ in parts]), site)
    assert np.array_equal(np.concatenate([b for _, b in parts], axis=1), post)


@pytest.mark.gpu
def test_c4_kernel_at_its_own_shape(gpu_backend):
    """1024 taxa x 131 072 binary sites, GTR + Gamma-4: the C4 default (tiled 2-state kernel) against the oracle."""
    from cybayes_b200.likelihood import _plan_for, engine_for
    from large_cases import SEED, _engine_inputs, _setup
    N, P, chunk = 1024, 131072, 16384
    aln, codes, leaves = _setup(N, P, 2, SEED, chunk)
    edges = aln.edge_order()
    tm = [oracle.prob_t("GTR", True, aln.pi, aln.tree, aln.er, r) for r in aln.rates]
    kids = [c for p, c in edges if p == aln.root]
    want, per_site, kept = oracle.mat_ml_scaled_codes(aln.pi, aln.root, codes, 2, None, edges, tm, N, chunk=chunk,
                                                      keep_nodes=tuple(c for c in kids if c > N))
    terms = _root_terms(aln.pi, aln.root, edges, tm, kept, lambda t: oracle.leaves_from_codes(codes[t - 1:t], 2)[1])
    from cybayes_b200 import likelihood
    likelihood.COMPRESS_MAX_SITES, saved = 0, likelihood.COMPRESS_MAX_SITES
    try:
        eng, _ = engine_for(leaves, 4)
    finally:
        likelihood.COMPRESS_MAX_SITES = saved
    plan = _plan_for(edges)
    _, _, pslots = _engine_inputs(eng, plan, aln.tree, tm, 4)
    lnl, site, post, _ = eng.eval_sites(None, plan.nodes, plan.children, pslots, aln.pi, categories=True)
    assert eng.n_patterns == P
    _check_against_oracle(site, post, lnl, per_site, terms)
    assert abs(lnl - want) <= 1e-11 * abs(want)


@pytest.mark.gpu
def test_deep_tree_gives_finite_site_terms(gpu_backend):
    """A 1300-taxon caterpillar that underflows the reference (every site's unscaled likelihood is 0): finite l,
    equal to the scaled oracle's."""
    from cybayes_b200.engine import Engine
    from cybayes_b200.likelihood import _Plan
    from large_cases import _engine_inputs
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
    tm = [oracle.prob_t("F81", True, pi, tree, None, r) for r in oracle.site_rates(0.5)]
    leaves = oracle.leaves_from_codes(codes, S)
    assert oracle.mat_ml(pi, root, leaves, edges, tm, n_sites, n_taxa)[0] == -np.inf
    per_site, terms = _oracle_sites(pi, root, leaves, edges, tm, n_sites, n_taxa)
    eng = Engine(codes, S, C)
    plan = _Plan(edges)
    _, _, pslots = _engine_inputs(eng, plan, tree, tm, C)
    lnl, site, post, _ = eng.eval_sites(None, plan.nodes, plan.children, pslots, pi, categories=True)
    _check_against_oracle(site, post, lnl, per_site, terms)
    eng.close()


@pytest.mark.gpu
def test_native_chain_site_lnl(golden_cases, gpu_backend, tmp_path):
    """narrow.phy F81: the accept / reject trace with sampling on is the recorded one; every row of the native
    .sitelnl sums to the chain's lnL; the native and Python drivers' files agree entry for entry."""
    from cybayes_b200 import likelihood
    from cybayes_b200.driver import run_chain
    from cybayes_b200.fastchain import run_chain_native
    from trace_checks import compare_trace
    rows, meta = load_trace("narrow_F81")
    n_gen, thin = 600, 50
    rec = []
    res = run_chain_native(NARROW, "F81", n_gen, thin, "bin", str(tmp_path / "n"), out=io.StringIO(), site_lnl=True,
                           on_generation=lambda i, cur, prop, p, mv, acc, st: rec.append((i, cur, prop, p, mv, acc)))
    compare_trace(rec, rows[:n_gen], meta, res["initial_lnL"], 1e-11)
    _, nat = _read_sitelnl(str(tmp_path / "n.sitelnl"))
    log = [line.split("\t") for line in open(str(tmp_path / "n.log")).read().splitlines()[1:]]
    assert len(nat) == len(log) == n_gen // thin
    for row, lr in zip(nat, log):
        assert abs(sum(row[1:]) - float(lr[1])) <= 1e-12 * abs(float(lr[1])), (row[0], lr)
    likelihood.reset_engines()
    run_chain(NARROW, "F81", n_gen, thin, "bin", str(tmp_path / "p"), out=io.StringIO(), site_lnl=True)
    _, py = _read_sitelnl(str(tmp_path / "p.sitelnl"))
    np.testing.assert_allclose(np.array(nat), np.array(py), rtol=1e-11, atol=0)
