"""CPU: host logic of the product (readers, leaf encoding, pattern compression, traversal
indexing, start state, proposals' random-number consumption, P-table bookkeeping, op-list
planning, the drivers) with the oracle-backed FakeEngine standing in for the CUDA engine."""
import hashlib
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

CASES = ["binary_F81", "twoStates_F81", "twoStates_JC", "narrow_F81", "narrow_JC", "narrow_GTR", "broad_F81",
         "phon_ringe_JC", "phon_ringe_F81", "phon_ringe_GTR", "ie42_JC", "ie42_GTR", "ielex2016_JC",
         "ielex_multistate_F81", "german_multistate_JC"]


def _digest(ll, n_taxa):
    h = hashlib.sha256()
    for k in range(1, n_taxa + 1):
        h.update(np.packbits(np.ascontiguousarray(ll[k]).astype(bool), axis=None).tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("name", CASES)
def test_readers_bit_exact(name, golden_cases):
    from cybayes_b200 import utils
    case = golden_cases[name]
    n, S, alphabet, site_dict, ll, taxa, n_sites = getattr(utils, case["reader"])(golden_io.data_path(case))
    assert (n, S, n_sites) == (case["n_taxa"], case["n_chars"], case["n_sites"])
    assert alphabet == case["alphabet"] and taxa == case["taxa"]
    assert _digest(ll, n) == case["leaf_digest"]            # 0/1 leaf matrices, bit for bit
    assert ll[1].shape == (S, n_sites) and ll[1].flags["C_CONTIGUOUS"] and ll[1].dtype == np.float64
    assert sorted(ll.keys()) == list(range(1, n + 1)) and len(ll) == n


def test_read_multi_phy_accepts_readphy_layout_and_rejects_garbage(golden_cases, tmp_path):
    from cybayes_b200 import utils
    case = golden_cases["ielex_multistate_F81"]
    a = utils.readMultiPhy(golden_io.data_path(case))     # the reference raises here (SURVEY F4)
    b = utils.readPhy(golden_io.data_path(case))
    assert a[2] == b[2] and np.array_equal(a[4].codes, b[4].codes)
    bad = tmp_path / "bad.phy"
    bad.write_text("2 3\nt1 0 1 0\nt2 011\n")
    with pytest.raises(ValueError, match="too many values to unpack"):
        utils.readBinaryPhy(str(bad))
    ragged = tmp_path / "ragged.phy"
    ragged.write_text("2 3\nt1 010\n\nt2 01\n")
    with pytest.raises((AssertionError, ValueError)):
        utils.readBinaryPhy(str(ragged))


def test_polymorphic_and_missing_cells(tmp_path):
    from cybayes_b200 import utils
    f = tmp_path / "poly.phy"
    f.write_text("3 4\nA\tx y x/y ?\nB\ty z - x/z\nC\tz/y x y z\n")
    n, S, alphabet, _, ll, taxa, n_sites = utils.readPhy(str(f))
    _, S2, alphabet2, _, ll2, _, _ = oracle.read_phylip(str(f), "readPhy")
    assert alphabet == alphabet2 == ["x", "y", "z"]
    for k in (1, 2, 3):
        assert np.array_equal(ll[k], ll2[k])
    assert ll.codes.dtype == np.uint8 and ll.codes.max() >= S   # ambiguity codes in use


def _py_patterns(codes):
    seen, weights, smap = {}, [], []
    for p in range(codes.shape[1]):
        key = codes[:, p].tobytes()
        if key not in seen:
            seen[key] = len(weights)
            weights.append(0)
        weights[seen[key]] += 1
        smap.append(seen[key])
    cols = [np.frombuffer(k, dtype=codes.dtype) for k in seen]
    return np.array(cols).T, np.array(weights, dtype=float), np.array(smap)


@pytest.mark.parametrize("name,n_patterns", [("narrow_F81", 943), ("broad_F81", 4377), ("binary_F81", None)])
def test_pattern_compression_bit_exact(name, n_patterns, golden_cases):
    from cybayes_b200 import utils
    from cybayes_b200.alignment import compress_patterns
    case = golden_cases[name]
    codes = getattr(utils, case["reader"])(golden_io.data_path(case))[4].codes
    pat, w, smap = compress_patterns(codes)
    pat2, w2, smap2 = _py_patterns(codes)
    assert np.array_equal(pat, pat2) and np.array_equal(w, w2) and np.array_equal(smap, smap2)
    assert w.sum() == codes.shape[1] and np.array_equal(pat[:, smap], codes)
    if n_patterns:
        assert pat.shape[1] == n_patterns      # SURVEY F2: 943 of 2351, 4377 of 5695


@pytest.mark.parametrize("name", ["binary_F81", "narrow_F81", "narrow_JC", "phon_ringe_GTR", "ie42_JC"])
def test_state_init_consumes_random_numbers_like_the_reference(name, golden_cases, fake_backend):
    from cybayes_b200 import config
    from cybayes_b200.driver import load_alignment
    from cybayes_b200.mcmc_gamma import get_siterates, state_init
    case = golden_cases[name]
    np.random.seed(1234)
    random.seed(1234)
    load_alignment(golden_io.data_path(case), case["dtype"], case["reader"])
    config.MODEL = case["model"]
    st = state_init()
    assert [[p, c, t] for (p, c), t in st["tree"].items()] == case["tree"]    # dict order and lengths
    assert st["root"] == case["root"] and st["srates"] == case["srates"]
    assert [list(e) for e in st["postorder"]] == case["postorder"]
    assert np.array_equal(np.asarray(st["pi"]), case["pi"])
    assert hashlib.sha256(np.asarray(st["rates"]).tobytes()).hexdigest() == case["rates_digest"]
    assert get_siterates(st["srates"]) == case["site_rates"]
    assert config.NORM_BETA == case["norm_beta"]


def _run_trace(name, n_gen, golden_cases, tmp_path, **kw):
    from cybayes_b200.driver import run_chain
    case = golden_cases[name]
    rec = []
    res = run_chain(golden_io.data_path(case), case["model"], n_gen, 1, case["dtype"], str(tmp_path / "run"),
                    out=io.StringIO(), on_generation=lambda i, cur, prop, p, mv, acc, st: rec.append(
                        (i, cur, prop, str(p), mv, acc)), **kw)
    return rec, res


@pytest.mark.parametrize("name,n_gen", [("binary_F81", 300), ("twoStates_JC", 300), ("narrow_F81", 250),
                                        ("phon_ringe_F81", 300), ("phon_ringe_GTR", 150)])
def test_driver_trace_on_fake_engine(name, n_gen, golden_cases, fake_backend, tmp_path):
    """Move sequence, proposed likelihoods and accept decisions equal the reference's recorded run."""
    rows, meta = load_trace(name)
    rec, res = _run_trace(name, n_gen, golden_cases, tmp_path)
    assert abs(res["initial_lnL"] - meta["init_lnL"]) <= 1e-12 * abs(meta["init_lnL"])
    for r, g in zip(rec, rows):
        assert (r[3], r[4]) == (g["param"], g["move"]), (r, g)
        assert abs(r[2] - float(g["proposed_ll"])) <= 1e-10 * abs(float(g["proposed_ll"])), (r, g)
        assert abs(r[1] - float(g["current_ll"])) <= 1e-10 * abs(float(g["current_ll"])), (r, g)
    log_rows = open(str(tmp_path / "run.log")).read().splitlines()[1:]
    assert [l.split("\t")[2:] for l in log_rows] == [[g["log_TL"], g["alpha"]] for g in rows[:n_gen]]


def test_fast_spr_is_the_same_chain(golden_cases, fake_backend, tmp_path):
    rec_a, _ = _run_trace("binary_F81", 300, golden_cases, tmp_path, fast_spr=False)
    n_ops_full = sum(e.n_ops for e in fake_backend.instances)
    fake_backend.instances.clear()
    from cybayes_b200 import likelihood
    likelihood.reset_engines()
    rec_b, _ = _run_trace("binary_F81", 300, golden_cases, tmp_path, fast_spr=True)
    n_ops_fast = sum(e.n_ops for e in fake_backend.instances)
    assert [(r[3], r[4], r[5]) for r in rec_a] == [(r[3], r[4], r[5]) for r in rec_b]
    assert all(abs(a[2] - b[2]) <= 1e-12 * abs(a[2]) for a, b in zip(rec_a, rec_b))
    assert n_ops_fast < n_ops_full


def test_unmodified_reference_driver_on_compat_modules(golden_cases, fake_backend, tmp_path, monkeypatch, capsys):
    """The reference's own script (byte-compiled, unmodified) imports `utils`, `config`, `mcmc_gamma`,
    `ML_gamma` from cybayes_b200/compat and produces its recorded per-generation output."""
    script = os.path.join(REPO, "oracle", "_ref", "mat_mcmc_gamma.code")
    if not os.path.exists(script):
        pytest.skip("no reference driver available (oracle/build_ref.sh)")
    monkeypatch.syspath_prepend(os.path.join(REPO, "cybayes_b200", "compat"))
    names = ("config", "utils", "mcmc_gamma", "ML_gamma", "mcmc", "ML")
    for m in names:
        monkeypatch.delitem(sys.modules, m, raising=False)
    case = golden_cases["narrow_F81"]
    n_gen = 200
    monkeypatch.setattr(sys, "argv", ["mat_mcmc_gamma.py", "-i", golden_io.data_path(case), "-m", "F81", "-n",
                                      str(n_gen), "-t", "1", "-d", "bin", "-o", str(tmp_path / "ref_run")])
    runpy.run_path(script, run_name="__main__")
    out = capsys.readouterr().out
    rows, _ = load_trace("narrow_F81")
    gens = [l.split("\t") for l in out.splitlines() if l.split("\t")[0].isdigit() and len(l.split("\t")) == 6]
    assert len(gens) == n_gen
    for f, g in zip(gens, rows):
        assert (f[4], f[5], f[3]) == (g["param"], g["move"], g["TL"]), (f, g)
        assert abs(float(f[2]) - float(g["proposed_ll"])) <= 1e-10 * abs(float(g["proposed_ll"]))
    for m in names:
        sys.modules.pop(m, None)


def test_pmat_table_lifetimes(fake_backend):
    """NNI aliasing: one slot referenced from two edges must survive deleting either key."""
    from cybayes_b200.subst import PMatTable, host_matrix
    eng = fake_backend(np.zeros((4, 8), dtype=np.uint8), 2, 4)
    block = eng.alloc_slots(3)
    t = PMatTable(eng, [(5, 1), (5, 2), (6, 5)], block)
    extra = host_matrix(eng, np.eye(2) * 0.5)
    slot = extra.slot
    t[5, 1] = extra
    t[6, 3] = t[5, 1].copy()
    del extra
    del t[5, 1]
    assert t._slots[6, 3] == slot and slot not in eng._free_slots.get(1, [])
    del t[6, 3]
    assert slot in eng._free_slots.get(1, [])          # last reference gone -> slot back in the pool
    assert (5, 2) in t and len(t) == 2 and list(t.keys()) == [(5, 2), (6, 5)]
    t2 = t.copy()
    del t
    assert block.base not in eng._free_slots.get(3, [])   # the copy keeps the block alive
    del t2, block
    assert eng._free_slots.get(3) is not None


def test_plan_orders_ops_like_the_reference_walk(golden_cases):
    from cybayes_b200.likelihood import _Plan
    case = golden_cases["binary_F81"]
    edges = [tuple(e) for e in case["postorder"]]
    plan = _Plan(edges)
    done, seen = [], {}
    for p, c in edges:                      # ML_gamma.pyx:24-36: a parent completes at its 2nd edge
        seen[p] = seen.get(p, 0) + 1
        if seen[p] == 2:
            done.append(p)
    assert plan.nodes.tolist() == done and plan.nodes[-1] == case["root"]
    for i, n in enumerate(plan.nodes.tolist()):
        assert tuple(plan.children[2 * i:2 * i + 2]) == plan.kids[n]
        for c in plan.kids[n]:
            assert c <= case["n_taxa"] or plan.index[c] < i      # children before parents


def test_non_gamma_surface(golden_cases, fake_backend):
    """mcmc / ML mirrors (single rate category): state_init + matML + cache_matML vs the oracle."""
    from cybayes_b200 import ML, config, mcmc
    from cybayes_b200.driver import load_alignment
    case = golden_cases["phon_ringe_F81"]
    np.random.seed(1234)
    random.seed(1234)
    load_alignment(golden_io.data_path(case), "multi")
    config.MODEL = "F81"
    st = mcmc.state_init()
    lnl, cache = ML.matML(st, config.TAXA, config.LEAF_LLMAT)
    _, _, _, _, ll, _, n_sites = oracle.read_phylip(golden_io.data_path(case), "readMultiPhy")
    tm = [oracle.prob_t("F81", False, np.asarray(st["pi"]), st["tree"], None, 1.0)]
    part = {}
    for p, c in st["postorder"]:
        v = tm[0][p, c].dot(ll[c] if c <= config.N_TAXA else part[c])
        part[p] = v if p not in part else part[p] * v
    want = np.sum(np.log(np.dot(np.asarray(st["pi"]), part[st["root"]])))       # ML.pyx:48
    assert abs(lnl - want) <= 1e-12 * abs(want)
    tree2, hr, pr, edge = mcmc.scale_edge(st["tree"].copy())
    st2 = dict(st, tree=tree2)
    st2["transitionMat"] = mcmc.get_edge_transition_mat(st["pi"], st["rates"], tree2[edge], st["transitionMat"], edge)
    path = mcmc.get_path2root(mcmc.adjlist2reverse_nodes_dict(st["tree"]), edge[1], st["root"])
    l2, _ = ML.cache_matML(st2, config.TAXA, config.LEAF_LLMAT, cache, path)
    tm2 = [oracle.prob_t("F81", False, np.asarray(st["pi"]), tree2, None, 1.0)]
    want2 = oracle.mat_ml(np.asarray(st["pi"]), st["root"], ll, st["postorder"], tm2 * 1, n_sites, config.N_TAXA, 1)[0]
    assert abs(l2 - want2) <= 1e-12 * abs(want2)


@pytest.mark.parametrize("name,fname,model,dtype,n_gen", [("ng_binary_F81", "binary.phy", "F81", "bin", 300),
                                                          ("ng_phon_ringe_JC", "phon_ringe.phy", "JC", "multi", 300)])
def test_unmodified_non_gamma_driver_on_compat_modules(name, fname, model, dtype, n_gen, fake_backend, tmp_path,
                                                       monkeypatch, capsys):
    """mat_mcmc.py (single-rate surface: mcmc + ML) unchanged, including its quirk of not refreshing
    the cache after accepted branch moves (mat_mcmc.py:141-152)."""
    from conftest import check_nongamma_trace, run_reference_script
    out = run_reference_script("mat_mcmc", ["-i", os.path.join(REPO, "tests", "golden", "data", fname), "-m", model,
                                            "-n", str(n_gen), "-t", "1", "-d", dtype, "-o", str(tmp_path / "ng")],
                               monkeypatch, capsys)
    check_nongamma_trace(out, name, 1e-10)


def test_siterates_direct_quantile_is_bit_identical():
    """get_siterates calls scipy.special.chdtri instead of chi2.isf (same function under ~100 us of argument
    checking): the four category rates must keep the reference's bits (mcmc_gamma.pyx:596-602)."""
    from scipy.special import gammainc
    from scipy.stats import chi2
    from cybayes_b200 import config
    from cybayes_b200.subst import get_siterates
    config.N_CATS = 4
    rng = np.random.default_rng(11)
    for a in np.concatenate([rng.uniform(0.01, 5, 3000), rng.uniform(5, 200, 500), [1e-3, 0.6863337793704655, 1000.0]]):
        alpha = float(np.float32(a))
        cut = [chi2.isf(1 - p, 2 * alpha) for p in np.arange(0.25, 1, 0.25)]
        cum = [gammainc(alpha + 1, c * alpha) for c in cut]
        want = [cum[0] * 4, (cum[1] - cum[0]) * 4, (cum[2] - cum[1]) * 4, (1.0 - cum[2]) * 4]
        got = get_siterates(a)
        assert [float(x) for x in got] == [float(x) for x in want], (a, got, want)


@pytest.mark.parametrize("name", ["narrow_F81", "phon_ringe_JC", "phon_ringe_GTR"])
def test_get_prob_t_all_equals_per_category_calls(name, golden_cases, fake_backend):
    """The restated driver's one-entry builder for all rate categories must give the matrices of the reference's
    per-category get_prob_t calls (mat_mcmc_gamma.py:147) and keep its shared slot block alive per table."""
    from cybayes_b200 import config
    from cybayes_b200.driver import load_alignment
    from cybayes_b200.subst import get_prob_t, get_prob_t_all
    case = golden_cases[name]
    load_alignment(golden_io.data_path(case), case["dtype"], case["reader"])
    config.MODEL, config.NORM_BETA = case["model"], case["norm_beta"]
    tree, pi, rates, edges, site_rates = golden_io.case_state(case)
    if rates is None:
        rates = np.ones(1)
    one_by_one = [get_prob_t(pi, tree, rates, r) for r in site_rates]
    together = get_prob_t_all(pi, tree, rates, site_rates)
    assert len(together) == len(one_by_one)
    for a, b in zip(one_by_one, together):
        assert list(a.keys()) == list(b.keys())
        for e in list(tree)[::7]:
            assert np.array_equal(np.asarray(a[e]), np.asarray(b[e]))
    eng = together[0].engine
    n = together[0]._block.n
    first = together.pop(0)
    del first
    assert together[0]._block.base not in eng._free_slots.get(n, [])   # still referenced by the other tables
    base = together[0]._block.base
    del together, a, b
    assert base in eng._free_slots.get(n, [])


def test_slot_tables_by_key_order_equal_slot_tables_by_lookup(golden_cases, fake_backend):
    """Full evaluations map a transition-matrix table onto the op order with one permutation per key order instead
    of one lookup per edge: device tables as built, host dicts in any insertion order, edited tables and dicts with
    foreign keys (which fall back to the lookups) must all give the per-edge result."""
    import random as pyrandom
    from cybayes_b200 import config, likelihood
    from cybayes_b200.driver import load_alignment
    from cybayes_b200.ML_gamma import matML
    from cybayes_b200.subst import get_edge_transition_mat, get_prob_t, get_prob_t_all
    case = golden_cases["narrow_F81"]
    load_alignment(golden_io.data_path(case), case["dtype"], case["reader"])
    config.MODEL, config.NORM_BETA = case["model"], case["norm_beta"]
    tree, pi, rates, edges, site_rates = golden_io.case_state(case)
    args = (config.N_SITES, config.N_TAXA, config.N_CATS)
    want = golden_io.oracle_lnl(case)
    plan = likelihood._plan_for(edges)
    eng, _ = likelihood.engine_for(config.LEAF_LLMAT, config.N_CATS)

    def by_lookup(tables):
        got, keep = likelihood._slot_matrix(eng, tables, plan.edge_keys)
        return got, keep

    tabs = get_prob_t_all(pi, tree, rates, site_rates)
    assert all(t.pristine() is not None for t in tabs)
    fast, _ = likelihood._slot_matrix(eng, tabs, plan.edge_keys, plan=plan)
    assert all(t.pristine() is not None for t in tabs)          # no dict was built on the way
    slow, _ = by_lookup(tabs)
    assert np.array_equal(fast, slow) and len(plan._perms) == 1
    lnl, _ = matML(pi, case["root"], config.LEAF_LLMAT, edges, tabs, *args)
    assert abs(lnl - want) <= 1e-11 * abs(want)
    # host dicts, shuffled insertion order, one order per category
    rng = pyrandom.Random(5)
    host = []
    for t in [get_prob_t(pi, tree, rates, r) for r in site_rates]:
        keys = list(tree)
        rng.shuffle(keys)
        host.append({e: np.array(t[e]) for e in keys})
    lnl, _ = matML(pi, case["root"], config.LEAF_LLMAT, edges, host, *args)
    assert abs(lnl - want) <= 1e-11 * abs(want)
    fast, keep1 = likelihood._slot_matrix(eng, host, plan.edge_keys, plan=plan)
    slow, keep2 = by_lookup(host)
    assert np.array_equal(eng.download_pmats(fast.T.ravel()), eng.download_pmats(slow.T.ravel()))
    # an edited table and a dict with a key the plan does not have take the per-edge route
    e = list(tree)[3]
    tabs[1][e] = get_edge_transition_mat(pi, rates, tree[e] * site_rates[1] * 1.5)
    assert tabs[1].pristine() is None
    host[2][(9999, 9998)] = np.eye(len(pi))
    mixed = [tabs[0], tabs[1], host[2], host[3]]
    fast, keep3 = likelihood._slot_matrix(eng, mixed, plan.edge_keys, plan=plan)
    slow, keep4 = by_lookup(mixed)
    assert np.array_equal(eng.download_pmats(fast.T.ravel()), eng.download_pmats(slow.T.ravel()))
    assert np.array_equal(fast[:, :2], slow[:, :2])
    bad = dict(host[3])
    del bad[e]
    bad[(9999, 9998)] = np.eye(len(pi))                           # right size, wrong edges
    with pytest.raises(KeyError):
        likelihood._slot_matrix(eng, [bad], plan.edge_keys, plan=plan)


def test_dirty_path_op_lists_are_cached_per_plan(golden_cases, fake_backend):
    """cache_matML keeps the op list of a dirty path with its plan: repeated branch moves on one edge reuse it, and the
    cached and the first evaluation agree."""
    from cybayes_b200 import config, likelihood
    from cybayes_b200.driver import load_alignment
    from cybayes_b200.mcmc_gamma import adjlist2reverse_nodes_dict, get_path2root, get_prob_t
    from cybayes_b200.ML_gamma import cache_matML, matML
    case = golden_cases["binary_F81"]
    load_alignment(golden_io.data_path(case), case["dtype"], case["reader"])
    config.MODEL, config.NORM_BETA = case["model"], case["norm_beta"]
    tree, pi, rates, edges, site_rates = golden_io.case_state(case)
    tmats = [get_prob_t(pi, tree, rates, r) for r in site_rates]
    args = (config.N_SITES, config.N_TAXA, config.N_CATS)
    lnl, cache = matML(pi, case["root"], config.LEAF_LLMAT, edges, tmats, *args)
    path = get_path2root(adjlist2reverse_nodes_dict(tree), list(tree)[3][1], case["root"])
    l1, _ = cache_matML(pi, case["root"], config.LEAF_LLMAT, cache, path, edges, tmats, *args)
    plan = likelihood._plan_for(edges)
    assert len(plan._paths) == 1
    l2, _ = cache_matML(pi, case["root"], config.LEAF_LLMAT, cache, path, edges, tmats, *args)
    assert len(plan._paths) == 1 and l1 == l2 == lnl


def test_large_shape_parity_bodies_dry_run(fake_backend, monkeypatch):
    """The bodies of the benchmark-shape GPU parity tests (tests/large_cases.py), run small on the oracle-backed fake
    engine: keeps the test logic itself (kept partials, dirty-path bookkeeping, slot tables) exercised on CPU."""
    import large_cases
    from cybayes_b200 import likelihood
    monkeypatch.setattr(likelihood, "COMPRESS_MAX_SITES", 0)
    large_cases.run_c4_shape(48, 512, 128)
    likelihood.reset_engines()
    large_cases.run_c5_shape(12, 256, 64, 128)


def test_hostgather_packs_like_bytes_join(tmp_path):
    """csrc/hostgather.c (optional CPython helper of the host-table route): same bytes as the bytes.join route, and a
    clean False -- never a partial success -- on anything that is not a plain float64 matrix or the expected key order."""
    import subprocess
    from cybayes_b200 import likelihood
    hg = likelihood._hostgather
    if hg is None:
        csrc = os.path.join(os.path.dirname(os.path.abspath(likelihood.__file__)), "csrc")
        if subprocess.run(["make", "-C", csrc, "../_hostgather.so"], capture_output=True).returncode != 0:
            pytest.skip("_hostgather cannot be built here")
        from cybayes_b200 import _hostgather as hg
    rng = np.random.default_rng(3)
    mats = [rng.random((3, 3)) for _ in range(50)]
    out = np.empty(50 * 9)
    assert hg.pack(mats, out) is True and out.tobytes() == b"".join(mats)
    assert hg.pack(tuple(mats), out) is True
    assert hg.pack([], np.empty(0)) is True
    for bad in (mats[0].T, mats[0].astype(np.float32), mats[0].tolist(), rng.random((3, 4)), mats[0][:, ::-1],
                mats[0].astype(">f8")):
        assert hg.pack(mats[:10] + [bad] + mats[11:], out) is False
    with pytest.raises(TypeError):
        hg.pack(mats, np.empty(50 * 9, dtype=np.float32))
    with pytest.raises(TypeError):
        hg.pack(mats, np.empty((50, 18))[:, ::2])
    keys = [(i, i + 100) for i in range(50)]
    table = dict(zip(keys, mats))
    out2 = np.empty(50 * 9)
    assert hg.pack_dict(table, keys, out2) is True and out2.tobytes() == out.tobytes()
    assert hg.pack_dict(table, [(int(a), int(b)) for a, b in keys], out2) is True          # equal, not identical, keys
    assert hg.pack_dict(table, keys[::-1], out2) is False                                    # other order
    assert hg.pack_dict(table, keys[:-1], out2) is False and hg.pack_dict(table, keys + [(1, 1)], out2) is False
    assert hg.pack_dict(dict(table, **{}), keys, np.empty(50 * 9 + 1)) is False              # size does not divide
    table[keys[7]] = mats[7].T
    assert hg.pack_dict(table, keys, out2) is False
    import collections
    assert hg.pack_dict(collections.OrderedDict(zip(keys, mats)), keys, out2) is False       # exact dicts only
    # the gather used by matML gives the same array with and without the module
    want = likelihood._gather_host_matrices(mats, 50, 3).copy()
    saved = likelihood._hostgather
    try:
        likelihood._hostgather = None
        assert np.array_equal(likelihood._gather_host_matrices(mats, 50, 3), want)
        likelihood._hostgather = hg
        assert np.array_equal(likelihood._gather_host_matrices(mats, 50, 3), want)
        odd = [m.astype(np.float32) for m in mats]                                           # general route
        assert np.allclose(likelihood._gather_host_matrices(odd, 50, 3), want, rtol=1e-6)
    finally:
        likelihood._hostgather = saved
