"""Metropolis-Hastings driver over the GPU likelihood engine.

A restatement of the reference's live Gamma driver (mat_mcmc_gamma.py:1-227) as a function:
same command line, same proposal mix, same random-number consumption (NumPy legacy global
generator for the move choice, Python ``random`` inside the moves and for the accept test),
same ``.log`` / ``.trees`` / stdout layout -- so for a fixed seed the accept/reject trace equals
the reference's, which tests/ check against traces recorded from the unmodified reference.
The reference's own script also runs unchanged on this package (cybayes_b200/compat).

What differs is only where the arithmetic happens: every likelihood and every P matrix comes
from the CUDA library.  With ``fast_spr`` an external-SPR proposal is scored by recomputing just
the two dirty node-to-root paths instead of the whole tree (the reference does a full pass,
mat_mcmc_gamma.py:167-169); the numbers are bit-identical because the same kernels see the same
operands.
"""
from __future__ import annotations

import argparse
from bisect import bisect_right
import random
import sys
import time
from collections import defaultdict

import numpy as np

from . import config, utils
from .ML_gamma import cache_matML, matML
from .subst import get_edge_transition_mats, get_prob_t_all
from .mcmc_gamma import (adjlist2newickBL, adjlist2nodes_dict, adjlist2reverse_nodes_dict, externalSPR,
                         get_edge_transition_mat, get_path2root, get_prob_t, get_siterates, mvDualSlider,
                         node_slider, rooted_NNI, scale_alpha, scale_edge, state_init)

READERS = {"bin": "readBinaryPhy", "multi": "readMultiPhy"}


def load_alignment(input_file, data_type, reader=None):
    """Fill the config blackboard from a Phylip file (mat_mcmc_gamma.py:20-31)."""
    fn = getattr(utils, reader or READERS[data_type])
    if config.LEAF_LLMAT is not None:      # a previous alignment of this process: free its device context
        from . import likelihood
        likelihood.drop_engine(config.LEAF_LLMAT)
    (config.N_TAXA, config.N_CHARS, config.ALPHABET, site_dict, config.LEAF_LLMAT, config.TAXA,
     config.N_SITES) = fn(input_file)
    config.IN_DTYPE = data_type
    config.N_NODES = 2 * config.N_TAXA - 1
    return site_dict


def move_table(model, n_rates=None, skip_degenerate_rates=False):
    """Parameter blocks, their weights and the moves of each block (mat_mcmc_gamma.py:65-84).
    With skip_degenerate_rates, a GTR model with a single exchangeability (binary data) gets no `rates` block: the
    reference proposes it anyway and dies in random.sample(range(1), 2) (mcmc_gamma.pyx:189, SURVEY F5); the default
    keeps that behaviour so the chain stays comparable with the reference up to its crash."""
    if model == "F81":
        params, w = ["pi", "tree", "bl", "srates"], [0.5, 3, 4, 0.5]
    elif model == "GTR" and skip_degenerate_rates and n_rates is not None and n_rates < 2:
        params, w = ["pi", "tree", "bl", "srates"], [0.5, 3, 4, 0.5]
    elif model == "GTR":
        params, w = ["pi", "rates", "tree", "bl", "srates"], [0.5, 0.5, 3, 4, 0.5]
    elif model == "JC":
        params, w = ["bl", "tree", "srates"], [4, 3, 0.5]
    else:
        raise ValueError(f"unknown model {model!r}")
    w = np.array(w, dtype=np.float64)
    tree_w = np.array([4, 1], dtype=np.float64)
    bl_w = np.array([3, 1], dtype=np.float64)
    moves = {"pi": [mvDualSlider], "rates": [mvDualSlider], "tree": [rooted_NNI, externalSPR],
             "bl": [scale_edge, node_slider], "srates": [scale_alpha]}
    return params, w / np.sum(w), moves, tree_w / np.sum(tree_w), bl_w / np.sum(bl_w)


def _spr_dirty_nodes(old_parent_of, new_tree, root):
    """Internal nodes whose partial changes under an external SPR: every node whose child set or
    child branch length changed, plus all their ancestors in the new tree."""
    new_parent_of = adjlist2reverse_nodes_dict(new_tree)
    dirty = set()
    for (p, c) in new_tree:
        if old_parent_of.get(c) != p:
            dirty.add(p)
    for c, p in old_parent_of.items():
        if new_parent_of.get(c) != p:
            dirty.add(p)
    out = set()
    for n in dirty:
        if n not in new_parent_of and n != root:
            continue
        out.add(n)
        while n != root:
            n = new_parent_of[n]
            out.add(n)
    return out


def spr_tables(tmats, tree_prop, pi, rates, site_rates):
    """Per-category P tables of the tree after an external SPR: the tables of the current tree with the three
    removed edges dropped and the three new ones built (same matrices as a full get_prob_t would give them)."""
    out = []
    for k, rate in enumerate(site_rates):
        t = tmats[k].copy()
        for e in [e for e in t.keys() if e not in tree_prop]:
            del t[e]
        for e, bl in tree_prop.items():
            if e not in t:
                t[e] = get_edge_transition_mat(pi, rates, bl * rate)
        out.append(t)
    return out


def open_site_lnl(output_file, n_columns):
    """<output_file>.sitelnl with its header: Iter, then the alignment columns 1..n_columns."""
    fh = open(output_file + ".sitelnl", "w")
    print("Iter", *range(1, n_columns + 1), sep="\t", file=fh)
    return fh


def write_site_lnl(fh, n_iter, site_lnl):
    """One sample: the generation, then the log-likelihood of every alignment column (%.17g: round-trips)."""
    fh.write(str(n_iter) + "\t" + "\t".join(["%.17g" % x for x in site_lnl.tolist()]) + "\n")


def run_chain(input_file, model, n_gen, thin, data_type, output_file, reader=None, seed=1234,
              out=sys.stdout, fast_spr=False, on_generation=None, diag=None, skip_degenerate_rates=False,
              site_lnl=False, ppc=0, ppc_seed=1):
    """Run the chain; returns a dict with the final state, counters and timings.  `diag` (a dict) receives, before
    each on_generation call, the acceptance test's two sides: diag["ll_ratio"] and diag["log_u"].  site_lnl: also
    write <output_file>.sitelnl, one row of per-column log-likelihoods per sample (the generations of .log), computed
    from the current cache without a random draw.  ppc: also write <output_file>.ppc, `ppc` posterior predictive
    replicates per sample (ppc.write_sample), simulated from Philox streams keyed on ppc_seed: no MT19937 draw."""
    if site_lnl:
        from .likelihood import refuse_sharded_site_lnl
        refuse_sharded_site_lnl()
    if ppc:
        from .ppc import refuse_sharded_ppc
        refuse_sharded_ppc()
    np.random.seed(seed)
    random.seed(seed)
    load_alignment(input_file, data_type, reader)
    config.N_GEN, config.THIN, config.MODEL = n_gen, thin, model

    print("Characters ", config.N_CHARS, file=out)
    print("TAXA ", config.TAXA, file=out)
    print("Number of TAXA ", config.N_TAXA, file=out)
    print("Alphabet ", config.ALPHABET, file=out)

    if model == "JC":
        config.NORM_BETA = config.N_CHARS / (config.N_CHARS - 1)  # overwritten by state_init (:580)

    state = state_init()
    site_rates = get_siterates(state["srates"])
    root = state["root"]
    leaves, n_sites, n_taxa, n_cats = config.LEAF_LLMAT, config.N_SITES, config.N_TAXA, config.N_CATS

    state["logLikehood"], cache = matML(state["pi"], root, leaves, state["postorder"], state["transitionMat"],
                                        n_sites, n_taxa, n_cats)
    parent_of = adjlist2reverse_nodes_dict(state["tree"])
    print("Initial Random Tree ", adjlist2newickBL(state["tree"], adjlist2nodes_dict(state["tree"]), root) + ";",
          sep="\t", file=out)
    print("Initial Likelihood ", state["logLikehood"], file=out)
    initial_lnl = state["logLikehood"]

    params_list, weights, moves_dict, tree_w, bl_w = move_table(model, len(state["rates"]), skip_degenerate_rates)
    moves_count, accepts_count = defaultdict(int), defaultdict(int)
    log_fh = open(output_file + ".log", "w")
    trees_fh = open(output_file + ".trees", "w")
    print("Iter", "LnL", "TL", "Alpha", sep="\t", file=log_fh)
    site_fh = open_site_lnl(output_file, n_sites) if site_lnl else None
    if site_fh is not None:
        from .likelihood import site_log_likelihoods
    reps = ppc_fh = None
    if ppc:
        from .ppc import Replicates, open_ppc, write_sample
        reps, ppc_fh = Replicates(leaves, n_cats), open_ppc(output_file)

    # np.random.choice(a, p=w) == a[cdf.searchsorted(random_sample(), 'right')] and np.random.choice(a) ==
    # a[randint(0, len(a))] draw for draw (legacy RandomState); the direct forms skip ~35 us of argument checks
    # per generation without changing the random stream (the recorded traces pin this).
    def _cdf(w):
        c = np.asarray(w, dtype=np.float64).cumsum()
        return (c / c[-1]).tolist()
    params_cdf, tree_cdf, bl_cdf = _cdf(weights), _cdf(tree_w), _cdf(bl_w)
    params_list = list(params_list)
    random_sample, randint = np.random.random_sample, np.random.randint

    t_start = time.perf_counter()
    for n_iter in range(1, n_gen + 1):
        pi_prop, rates_prop = state["pi"].copy(), state["rates"].copy()
        tree_prop, order_prop = state["tree"], state["postorder"]
        hr, pr_ratio = 0.0, 0.0

        param = params_list[bisect_right(params_cdf, random_sample())]
        if param == "tree":
            move = moves_dict[param][bisect_right(tree_cdf, random_sample())]
        elif param == "bl":
            move = moves_dict[param][bisect_right(bl_cdf, random_sample())]
        else:
            move = moves_dict[param][randint(0, len(moves_dict[param]))]
        name = move.__name__
        moves_count[param, name] += 1

        tmats = state["transitionMat"]
        undo = []          # (category, edge, previous handle or None) to restore on rejection
        prop_tmats = None
        proposed_cache = None   # a rejected proposal's partials go back to the pool before the next evaluation
        if param in ("pi", "rates"):
            new_param, hr = move(state[param].copy())
            if param == "pi":
                pi_prop = new_param
            else:
                rates_prop = new_param
        elif param == "bl":
            if name == "scale_edge":
                tree_prop, hr, pr_ratio, edge = move(state["tree"].copy())
                changed = [edge]
            else:
                tree_prop, hr, pr_ratio, edge, upper = move(state["tree"].copy(), root)
                changed = [edge, upper]
            dirty = get_path2root(parent_of, edge[1], root)
        elif param == "tree":
            if name == "rooted_NNI":
                tree_prop, order_prop, hr, dirty, (a, b, src, tgt) = move(state["tree"].copy(), root)
            else:
                tree_prop, order_prop, hr = move(state["tree"].copy(), root)
        else:  # srates
            new_param, hr, pr_ratio = move(state["srates"])
            saved_rates = site_rates[:]
            site_rates = get_siterates(new_param)

        if param == "bl":
            new_p = iter(get_edge_transition_mats(pi_prop, rates_prop,
                                                  [tree_prop[e] * rate for rate in site_rates for e in changed]))
            for k in range(len(site_rates)):
                for e in changed:
                    undo.append((k, e, tmats[k][e]))
                    tmats[k][e] = next(new_p)
            proposed_ll, proposed_cache = cache_matML(pi_prop, root, leaves, cache, dirty, state["postorder"], tmats,
                                                      n_sites, n_taxa, n_cats)
        elif name == "rooted_NNI":
            for k in range(len(site_rates)):
                tmats[k][a, tgt], tmats[k][b, src] = tmats[k][b, tgt].copy(), tmats[k][a, src].copy()
            proposed_ll, proposed_cache = cache_matML(pi_prop, root, leaves, cache, dirty, order_prop, tmats,
                                                      n_sites, n_taxa, n_cats)
        elif name == "externalSPR" and fast_spr:
            dirty_set = _spr_dirty_nodes(parent_of, tree_prop, root)
            prop_tmats = spr_tables(tmats, tree_prop, pi_prop, rates_prop, site_rates)
            if dirty_set:
                proposed_ll, proposed_cache = cache_matML(pi_prop, root, leaves, cache, list(dirty_set), order_prop,
                                                          prop_tmats, n_sites, n_taxa, n_cats)
            else:  # the move was a no-op (hastings 0.0 branches): same tree, same likelihood
                proposed_ll, proposed_cache = cache_matML(pi_prop, root, leaves, cache, [root], order_prop,
                                                          prop_tmats, n_sites, n_taxa, n_cats)
        else:
            prop_tmats = get_prob_t_all(pi_prop, tree_prop, rates_prop, site_rates)
            proposed_ll, proposed_cache = matML(pi_prop, root, leaves, order_prop, prop_tmats, n_sites, n_taxa, n_cats)

        current_ll = state["logLikehood"]
        ll_ratio = proposed_ll - current_ll + pr_ratio
        ll_ratio += hr
        log_u = np.log(random.random())
        accepted = bool(log_u <= ll_ratio)
        if diag is not None:
            diag["ll_ratio"], diag["log_u"] = float(ll_ratio), float(log_u)
        if accepted:
            if param == "bl":
                state["tree"] = tree_prop
            elif param == "tree":
                state["tree"], state["postorder"] = tree_prop, order_prop
                parent_of = adjlist2reverse_nodes_dict(tree_prop)
            elif param == "pi":
                state["pi"] = pi_prop
            elif param == "rates":
                state["rates"] = rates_prop
            else:
                state["srates"] = new_param
            if prop_tmats is not None:
                state["transitionMat"] = prop_tmats
            if name == "rooted_NNI":
                for k in range(len(tmats)):
                    del tmats[k][a, src], tmats[k][b, tgt]
            state["logLikehood"] = proposed_ll
            cache = proposed_cache
            accepts_count[param, name] += 1
        else:
            if param == "srates":
                site_rates = saved_rates[:]
            elif param == "bl":
                for k, e, handle in undo:
                    tmats[k][e] = handle
            elif name == "rooted_NNI":
                for k in range(len(tmats)):
                    del tmats[k][a, tgt], tmats[k][b, src]

        if on_generation is not None:
            on_generation(n_iter, current_ll, proposed_ll, param, name, accepted, state)
        if n_iter % thin == 0:
            TL = sum(state["tree"].values())
            sampled = adjlist2newickBL(state["tree"], adjlist2nodes_dict(state["tree"]), root) + ";"
            print(n_iter, current_ll, proposed_ll, TL, param, name, sep="\t", file=out)
            print(n_iter, state["logLikehood"], TL, state["srates"], sep="\t", file=log_fh)
            print(n_iter, sampled, sep="\t", file=trees_fh)
            if site_fh is not None:
                write_site_lnl(site_fh, n_iter, site_log_likelihoods(state["pi"], root, leaves, state["postorder"],
                                                                     state["transitionMat"], cache=cache)[1])
            if reps is not None:
                write_sample(ppc_fh, reps, n_iter, n_iter // thin - 1, state, model, ppc, ppc_seed)
    elapsed = time.perf_counter() - t_start
    log_fh.close()
    trees_fh.close()
    if site_fh is not None:
        site_fh.close()
    if reps is not None:
        ppc_fh.close()
        reps.close()
    for k, v in moves_count.items():
        print(k, accepts_count[k], v, file=out)
    return {"state": state, "initial_lnL": initial_lnl, "moves": dict(moves_count), "accepts": dict(accepts_count),
            "seconds": elapsed, "gens_per_sec": n_gen / elapsed if elapsed > 0 else float("inf")}


def main(argv=None):
    ap = argparse.ArgumentParser(description="CyBayes-compatible MCMC on the B200 likelihood engine")
    ap.add_argument("-i", "--input_file", type=str, required=True)
    ap.add_argument("-m", "--model", type=str, required=True, help="JC/F81/GTR")
    ap.add_argument("-n", "--n_gen", type=int, required=True)
    ap.add_argument("-t", "--thin", type=int, required=True)
    ap.add_argument("-d", "--data_type", type=str, required=True, help="bin / multi")
    ap.add_argument("-o", "--output_file", type=str, required=True)
    ap.add_argument("--reader", type=str, default=None, help="override the reader (e.g. readPhy)")
    ap.add_argument("--fast-spr", action="store_true", help="dirty-path scoring of external SPR proposals")
    ap.add_argument("--native", action="store_true", help="run the generation loop inside the library (same trace)")
    ap.add_argument("--skip-degenerate-rates", action="store_true",
                    help="GTR on binary data: do not propose the single exchangeability (the reference crashes there)")
    ap.add_argument("--site-lnl", action="store_true",
                    help="also write <output>.sitelnl: per-column log-likelihoods at every sample (WAIC / LOO input)")
    ap.add_argument("--ppc", type=int, default=0, metavar="N",
                    help="also write <output>.ppc: N posterior predictive replicates per sample (lnL and multinomial T)")
    ap.add_argument("--ppc-seed", type=int, default=1, help="seed of the replicates' Philox streams (0 .. 2^64 - 1)")
    a = ap.parse_args(argv)
    if a.ppc < 0:
        ap.error("--ppc: the number of replicates per sample cannot be negative")
    if not 0 <= a.ppc_seed < 1 << 64:
        ap.error("--ppc-seed must be in 0 .. 2^64 - 1")
    if a.ppc:
        from .ppc import refuse_sharded_ppc
        try:
            refuse_sharded_ppc()
        except ValueError as e:
            ap.error(f"--ppc: {e}")
    if a.site_lnl:
        from .likelihood import refuse_sharded_site_lnl
        try:
            refuse_sharded_site_lnl()
        except ValueError as e:
            ap.error(f"--site-lnl: {e}")
    if a.native:
        from .fastchain import run_chain_native
        res = run_chain_native(a.input_file, a.model, a.n_gen, a.thin, a.data_type, a.output_file, reader=a.reader,
                               skip_degenerate_rates=a.skip_degenerate_rates, site_lnl=a.site_lnl, ppc=a.ppc,
                               ppc_seed=a.ppc_seed)
    else:
        res = run_chain(a.input_file, a.model, a.n_gen, a.thin, a.data_type, a.output_file, reader=a.reader,
                        fast_spr=a.fast_spr, skip_degenerate_rates=a.skip_degenerate_rates, site_lnl=a.site_lnl,
                        ppc=a.ppc, ppc_seed=a.ppc_seed)
    print(f"# {res['gens_per_sec']:.1f} generations/s", file=sys.stderr)


if __name__ == "__main__":
    main()
