"""TEST INFRASTRUCTURE: load the committed golden cases (tests/golden/cases.json) and rebuild, for
one case, the inputs both sides need: the alignment through the oracle's reader restatement, the
start tree / pi / rates / category rates exactly as recorded from the unmodified reference."""
import json
import os

import numpy as np

import pruning_oracle as oracle

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, "tests", "golden")


def load_cases():
    with open(os.path.join(GOLDEN, "cases.json")) as fh:
        return {c["name"]: c for c in json.load(fh)["cases"]}


def data_path(case):
    return os.path.join(GOLDEN, "data", case["file"])


def case_state(case):
    """(tree dict in recorded insertion order, pi, rates or None, edge order, site rates)."""
    tree = {(p, c): t for p, c, t in case["tree"]}
    edges = [tuple(e) for e in case["postorder"]]
    rates = None if case["rates"] is None else np.array(case["rates"])
    return tree, np.array(case["pi"]), rates, edges, list(case["site_rates"])


def oracle_lnl(case, tree=None, gtr_via="expm", scaled=False):
    """lnL of the case's start state (or of `tree`) computed by the NumPy oracle end to end."""
    tree0, pi, rates, edges, site_rates = case_state(case)
    tree = tree0 if tree is None else tree
    _, S, _, _, ll, _, n_sites = oracle.read_phylip(data_path(case), case["reader"])
    tm = [oracle.prob_t(case["model"], case["dtype"] == "bin", pi, tree, rates, r, beta=case["norm_beta"],
                        gtr_via=gtr_via) for r in site_rates]
    if scaled:
        return oracle.mat_ml_scaled(pi, case["root"], ll, edges, tm, n_sites, case["n_taxa"])
    return oracle.mat_ml(pi, case["root"], ll, edges, tm, n_sites, case["n_taxa"])[0]


RANDOM_VECTORS = os.path.join(GOLDEN, "random_inputs.npz")


def random_inputs():
    """The seeded random cases of the oracle-against-reference check: for (S, model) in four settings, an 11-taxon
    random-join tree with Exp(0.1) branch lengths, pi, exchangeabilities, the F81 beta and 57 sites of leaf columns
    (state S = all ones, i.e. missing)."""
    rng = np.random.default_rng(5)
    for S, model, dtype in ((2, "F81", "bin"), (5, "F81", "multi"), (5, "JC", "multi"), (4, "GTR", "multi")):
        n_taxa, n_sites = 11, 57
        nodes, nxt, tree = list(range(1, n_taxa + 1)), n_taxa + 1, {}
        while len(nodes) > 1:
            a = nodes.pop(int(rng.integers(len(nodes))))
            b = nodes.pop(int(rng.integers(len(nodes))))
            tree[nxt, a] = float(rng.exponential(0.1))
            tree[nxt, b] = float(rng.exponential(0.1))
            nodes.append(nxt)
            nxt += 1
        pi = rng.dirichlet(np.ones(S)) if model != "JC" else np.repeat(1.0 / S, S)
        er = rng.dirichlet(np.ones(S * (S - 1) // 2))
        eye = np.vstack([np.eye(S), np.ones(S)])
        ll = {t: np.ascontiguousarray(eye[rng.integers(0, S + 1, n_sites)].T) for t in range(1, n_taxa + 1)}
        yield {"S": S, "model": model, "dtype": dtype, "n_taxa": n_taxa, "n_sites": n_sites, "tree": tree,
               "root": nxt - 1, "pi": pi, "er": er, "beta": 1 / (1 - np.dot(pi, pi)), "ll": ll}


def random_vectors(i, case, edges, site_rates, tmats, lnl, path, lnl_dirty):
    """Entries of tests/golden/random_inputs.npz for random case i: edge order, category rates, P(t r_k) of every
    edge (categories x edges in the tree's insertion order), matML lnL, the dirty path from taxon 3 and the
    cache_matML lnL along it."""
    return {f"{i}_edges": np.array(edges, dtype=np.int64), f"{i}_site_rates": np.array(site_rates, dtype=np.float64),
            f"{i}_pmats": np.array([[np.asarray(t[e]) for e in case["tree"]] for t in tmats], dtype=np.float64),
            f"{i}_lnL": np.array(lnl, dtype=np.float64), f"{i}_path": np.array(path, dtype=np.int64),
            f"{i}_lnL_dirty": np.array(lnl_dirty, dtype=np.float64)}
