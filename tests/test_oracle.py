"""CPU: the NumPy oracle against the golden vectors recorded from the unmodified reference, and
against the compiled reference itself (oracle/_ref) when it is present."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

import golden_io
import pruning_oracle as oracle
from conftest import REPO

FAST = ["binary_F81", "twoStates_F81", "twoStates_JC", "narrow_F81", "narrow_GTR", "phon_ringe_JC", "phon_ringe_F81",
        "phon_ringe_GTR", "ie42_JC", "ielex_multistate_F81"]


def _leaf_digest(ll, n_taxa):
    h = hashlib.sha256()
    for k in range(1, n_taxa + 1):
        h.update(np.packbits(np.ascontiguousarray(ll[k]).astype(bool), axis=None).tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("name", FAST)
def test_oracle_reproduces_reference_vectors(name, golden_cases):
    case = golden_cases[name]
    n_leaves, S, alphabet, _, ll, taxa, n_sites = oracle.read_phylip(golden_io.data_path(case), case["reader"])
    # integer artefacts: exact
    assert (n_leaves, S, n_sites) == (case["n_taxa"], case["n_chars"], case["n_sites"])
    assert alphabet == case["alphabet"] and taxa == case["taxa"]
    assert _leaf_digest(ll, n_leaves) == case["leaf_digest"]
    tree, pi, rates, edges, site_rates = golden_io.case_state(case)
    assert oracle.edge_order(tree, case["root"], n_leaves) == edges
    np.testing.assert_array_equal(oracle.site_rates(case["srates"]), site_rates)
    if case["model"] == "F81":
        assert oracle.f81_beta(pi) == case["norm_beta"]
    # P(t) and likelihood
    tm = [oracle.prob_t(case["model"], case["dtype"] == "bin", pi, tree, rates, r, beta=case["norm_beta"])
          for r in site_rates]
    for key, mats in case["pmat_sample"].items():
        e = tuple(int(x) for x in key.split(","))
        for k, ref in enumerate(mats):
            if isinstance(ref, dict):
                assert np.array_equal(tm[k][e][0], ref["row0"]) and np.array_equal(np.diag(tm[k][e]), ref["diag"])
            else:
                assert np.array_equal(tm[k][e], np.array(ref))
    lnl, cache = oracle.mat_ml(pi, case["root"], ll, edges, tm, n_sites, n_leaves)
    assert abs(lnl - case["lnL"]) <= 1e-14 * abs(case["lnL"])
    for node, sums in case["partial_sums"].items():
        np.testing.assert_allclose([cache[k][int(node)].sum() for k in range(4)], sums, rtol=1e-13)
    scaled = oracle.mat_ml_scaled(pi, case["root"], ll, edges, tm, n_sites, n_leaves)
    assert abs(scaled - case["lnL"]) <= 1e-13 * abs(case["lnL"])
    parents = oracle.parent_of(tree)
    for d in case["dirty"]:
        e = tuple(d["edge"])
        assert oracle.path_to_root(parents, e[1], case["root"]) == d["path"]
        saved = [tm[k][e] for k in range(4)]
        Q = oracle.gtr_q(rates, pi) if case["model"] == "GTR" else None
        for k, r in enumerate(site_rates):
            tm[k][e] = oracle.p_matrix(case["model"], case["dtype"] == "bin", pi, rates,
                                       oracle.f81_beta(pi) if case["model"] == "F81" else case["norm_beta"],
                                       d["new_t"] * r, Q=Q)
        l2, _ = oracle.cache_mat_ml(pi, case["root"], ll, cache, d["path"], edges, tm, n_sites, n_leaves)
        assert abs(l2 - d["lnL"]) <= 1e-14 * abs(d["lnL"])
        for k in range(4):
            tm[k][e] = saved[k]


def test_scaled_oracle_survives_where_the_reference_underflows():
    rng = np.random.default_rng(3)
    n_taxa, n_sites = 1300, 20
    tree, prev, nxt = {}, 1, n_taxa + 1
    for tip in range(2, n_taxa + 1):
        tree[nxt, prev] = 0.6
        tree[nxt, tip] = 0.6
        prev, nxt = nxt, nxt + 1
    root = nxt - 1
    kids = oracle.children_of(tree)
    order, stack = [], [root]
    while stack:
        nd = stack.pop()
        x, y = kids[nd]
        order += [(nd, x), (nd, y)]
        stack += [c for c in (y, x) if c > n_taxa]
    edges = order[::-1]
    pi = np.array([0.4, 0.6])
    eye = np.eye(2)
    ll = {t: np.ascontiguousarray(eye[rng.integers(0, 2, n_sites)].T) for t in range(1, n_taxa + 1)}
    tm = [oracle.prob_t("F81", True, pi, tree, None, r) for r in oracle.site_rates(0.5)]
    assert oracle.mat_ml(pi, root, ll, edges, tm, n_sites, n_taxa)[0] == -np.inf
    total, per_site = oracle.mat_ml_scaled(pi, root, ll, edges, tm, n_sites, n_taxa, site_lnl=True)
    assert np.isfinite(total) and (per_site < -709).all()


def test_gtr_eigen_route_matches_expm():
    rng = np.random.default_rng(11)
    for S in (2, 6, 23):
        pi = rng.dirichlet(np.full(S, 3.0))
        er = rng.dirichlet(np.ones(S * (S - 1) // 2))
        for d in (1e-4, 0.02, 0.5, 3.0):
            a = oracle.p_matrix("GTR", False, pi, er, None, d, gtr_via="expm")
            b = oracle.p_matrix("GTR", False, pi, er, None, d, gtr_via="eig")
            np.testing.assert_allclose(b, a, rtol=5e-10, atol=1e-15)


def _assert_same_vectors(got, want):
    keys = sorted(k for k in want if k != "source")
    assert sorted(k for k in got if k != "source") == keys
    for k in keys:
        assert got[k].dtype == want[k].dtype and np.array_equal(got[k], want[k]), k


def test_oracle_against_compiled_reference_on_random_inputs(tmp_path):
    """Seeded random trees and data (golden_io.random_inputs): the oracle's edge order, category rates, P(t) of every
    edge, matML and cache_matML equal, bit for bit, the vectors stored in tests/golden/random_inputs.npz
    (make_golden.py --random-inputs).  Its `source` entry says what computed them: "oracle" means the oracle itself,
    recorded while it had none of its own changes since this test held it bit-equal to the compiled reference on these
    inputs (DESIGN.md section 4), so the stored file pins that agreement.  Where the compiled reference is built
    (oracle/_ref) it is run again, in a fresh interpreter so that its top-level module names do not leak into this
    one, and must reproduce the stored vectors too."""
    want = dict(np.load(golden_io.RANDOM_VECTORS))
    got = {}
    for i, c in enumerate(golden_io.random_inputs()):
        tree, root, pi, ll, N, P = c["tree"], c["root"], c["pi"], c["ll"], c["n_taxa"], c["n_sites"]
        edges = oracle.edge_order(tree, root, N)
        rates = oracle.site_rates(0.8)
        tm = [oracle.prob_t(c["model"], c["dtype"] == "bin", pi, tree, c["er"], r, beta=c["beta"]) for r in rates]
        lnl, cache = oracle.mat_ml(pi, root, ll, edges, tm, P, N)
        path = oracle.path_to_root(oracle.parent_of(tree), 3, root)
        l2, _ = oracle.cache_mat_ml(pi, root, ll, cache, path, edges, tm, P, N)
        assert l2 == lnl
        got.update(golden_io.random_vectors(i, c, edges, rates, tm, lnl, path, l2))
    _assert_same_vectors(got, want)
    if os.path.exists(os.path.join(REPO, "oracle", "_ref")):
        out = tmp_path / "reference.npz"
        res = subprocess.run([sys.executable, os.path.join(REPO, "tests", "golden", "make_golden.py"), "--random-inputs",
                              str(out), "reference"], cwd=REPO, capture_output=True, text=True)
        assert res.returncode == 0, res.stderr[-2000:]
        _assert_same_vectors(dict(np.load(out)), want)
