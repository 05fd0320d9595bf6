"""Posterior predictive checks (Gelman, Meng & Stern 1996; Bollback 2002): does the model fit the data at all?

At a sample of the chain, ``Replicates.draw`` simulates a replicate alignment under the sampled tree and parameters on
the GPU (cb_simulate) and returns two discrepancy statistics of it: its log-likelihood under the same state, and the
multinomial statistic T = sum_i n_i ln n_i - n ln n over its unique columns.  The observed data's values are the
sample's lnL and ``Replicates.T_obs``.  The drivers' ``--ppc N`` writes N replicates per sample to <output>.ppc, and
``python -m cybayes_b200.ppc out.ppc`` reports, per statistic, how often the replicate falls at or below the observed
value (the posterior predictive p-value; values near 0 or 1 say the model does not reproduce that feature of the data).

The replicate context holds the observed columns uncompressed (weights 1), so a replicate keeps the observed
alignment's missing-data and polymorphism layout cell for cell: cb_simulate writes only cells that hold a state.
"""
from __future__ import annotations

import argparse
import math
import os
import sys

import numpy as np

from . import config, likelihood, subst
from .alignment import LeafMatrices, compress_patterns, pattern_weights_gpu
from .engine import Engine

PPC_HEADER = ("Iter", "Replicate", "LnL_obs", "LnL_rep", "T_obs", "T_rep")


def refuse_sharded_ppc():
    """A replicate is simulated, compressed and scored whole; a site-sharded rank holds only its slice of the columns."""
    if os.environ.get("CYBAYES_SHARD", "0") == "1":
        raise ValueError("posterior predictive checks are not available with CYBAYES_SHARD=1: each rank holds only its "
                         "slice of the alignment's columns")


def multinomial_statistic(weights):
    """T = sum_i n_i ln n_i - n ln n over the multiplicities n_i of the unique columns, n = sum_i n_i (Bollback 2002):
    the log-likelihood of the columns under the saturated multinomial model."""
    w = np.asarray(weights, dtype=np.float64)
    n = float(w.sum())
    return float(np.sum(w * np.log(w)) - n * math.log(n))


def column_weights(codes):
    """Multiplicities of the unique columns of `codes`, through the pattern-compression route the likelihood takes for
    an alignment of that length (host NumPy, or cb_compress_patterns on the GPU for long ones, whose pattern columns
    are not gathered: T needs only their multiplicities)."""
    host_max = likelihood.COMPRESS_MAX_SITES or 250000
    if codes.shape[1] > host_max and likelihood.COMPRESS_GPU and likelihood._engine_factory is Engine:
        return pattern_weights_gpu(codes)[0]
    return compress_patterns(codes)[1]


class Replicates:
    """Replicate alignments of one observed alignment (`leaves`, as config.LEAF_LLMAT) under sampled states.  Owns a
    context built from the observed uncompressed columns; every draw overwrites its state cells."""

    def __init__(self, leaves, n_cats):
        refuse_sharded_ppc()
        if isinstance(leaves, LeafMatrices):
            codes, S, amb = leaves.codes, leaves.n_states, leaves.amb_sets
        else:
            codes, S, amb = likelihood._codes_from_dense(leaves, len(leaves))
        self.n_cats = int(n_cats)
        self.engine = likelihood._engine_factory(np.ascontiguousarray(codes), S, self.n_cats, amb)
        # T of the observed data from the pattern weights the likelihood's context already holds
        main, site_map = likelihood.engine_for(leaves, self.n_cats)
        self.T_obs = multinomial_statistic(main.weights if site_map is not None else column_weights(codes))

    def _tables(self, state, model):
        """The state's P matrices, built in this context through the substitution models' device route (all edges x
        categories in one queue entry, as get_prob_t_all builds them), with the edge list in preorder for cb_simulate
        and the op list of a full pass over the same slots."""
        eng, C = self.engine, self.n_cats
        tree, root = state["tree"], int(state["root"])
        edges = list(tree)
        n_e = len(edges)
        block = eng.alloc_slots(n_e * C)
        site_rates = subst.get_siterates(state["srates"])
        d = np.multiply.outer(np.array(site_rates, dtype=np.float64),
                              np.fromiter(tree.values(), dtype=np.float64, count=n_e)).ravel()
        pi = np.asarray(state["pi"], dtype=np.float64)
        beta = subst.f81_beta(pi) if model == "F81" else config.NORM_BETA
        subst._queue(eng, model, config.IN_DTYPE == "bin", pi, state["rates"],
                     np.arange(block.base, block.base + block.n, dtype=np.int32), d, beta)
        out_edges = {}
        for i, (p, _) in enumerate(edges):
            out_edges.setdefault(p, []).append(i)
        order, stack = [], [root]
        while stack:
            for i in out_edges.get(stack.pop(), ()):
                order.append(i)
                stack.append(edges[i][1])
        if len(order) != n_e:
            raise ValueError("the state's tree is not connected to its root")
        cat = np.arange(C, dtype=np.int32)[None, :] * n_e + block.base
        pre = np.array(order, dtype=np.int32)
        parents = np.array([edges[i][0] for i in order], dtype=np.int32)
        children = np.array([edges[i][1] for i in order], dtype=np.int32)
        plan = likelihood._Plan([edges[i] for i in reversed(order)])   # children before parents
        where = {e: i for i, e in enumerate(edges)}
        ops = np.array([where[e] for e in plan.edge_keys], dtype=np.int32)
        return block, pi, root, (parents, children, pre[:, None] + cat), (plan, ops[:, None] + cat)

    def lnl(self, state, model):
        """lnL of the columns this context holds now under `state` (before the first draw: the observed columns)."""
        block, pi, _, _, (plan, pslots) = self._tables(state, model)
        lnl, _ = self.engine.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=False)
        return float(lnl)

    def draw(self, state, model, seed, replicate):
        """One replicate under `state` (tree, root, pi, rates, srates): (lnL_rep, T_rep)."""
        block, pi, root, (parents, children, ps_sim), (plan, ps_eval) = self._tables(state, model)
        codes = self.engine.simulate(parents, children, ps_sim, pi, root, seed, replicate)
        lnl, _ = self.engine.eval(None, plan.nodes, plan.children, ps_eval, pi, want_snapshot=False)
        return float(lnl), multinomial_statistic(column_weights(codes))

    def close(self):
        self.engine.close()


def open_ppc(output_file):
    """<output_file>.ppc with its header."""
    fh = open(output_file + ".ppc", "w")
    print(*PPC_HEADER, sep="\t", file=fh)
    return fh


def write_sample(fh, reps, n_iter, sample, state, model, n_rep, seed):
    """The n_rep replicates of one sample (the sample-th, from 0); replicate ids sample * n_rep + j.  Each row:
    generation, replicate id, lnL_obs (the sample's lnL as in .log), lnL_rep, T_obs, T_rep."""
    lnl_obs = float(state["logLikehood"])
    for j in range(n_rep):
        rid = sample * n_rep + j
        lnl_rep, t_rep = reps.draw(state, model, seed, rid)
        fh.write("%d\t%d\t%.17g\t%.17g\t%.17g\t%.17g\n" % (n_iter, rid, lnl_obs, lnl_rep, reps.T_obs, t_rep))


def read_ppc(path):
    """The rows of a .ppc file as a (n_rows, 6) float64 array."""
    with open(path) as fh:
        head = fh.readline().rstrip("\n").split("\t")
        if tuple(head) != PPC_HEADER:
            raise ValueError(f"{path}: not a .ppc file (header {head})")
        rows = [[float(x) for x in line.split("\t")] for line in fh if line.strip()]
    return np.array(rows, dtype=np.float64).reshape(-1, len(PPC_HEADER))


def summary(path, burnin=0):
    """Per statistic ('lnL', 'T'): the posterior predictive p-value P(replicate <= observed) over the replicates of the
    samples after generation `burnin`, the observed mean and the replicate mean."""
    rows = read_ppc(path)
    rows = rows[rows[:, 0] > burnin]
    if rows.shape[0] == 0:
        raise ValueError(f"{path}: no replicate after generation {burnin}")
    out = {}
    for name, obs, rep in (("lnL", rows[:, 2], rows[:, 3]), ("T", rows[:, 4], rows[:, 5])):
        out[name] = {"p": float(np.mean(rep <= obs)), "observed_mean": float(np.mean(obs)),
                     "replicate_mean": float(np.mean(rep)), "replicates": int(rows.shape[0])}
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description="posterior predictive p-values of a .ppc file")
    ap.add_argument("path")
    ap.add_argument("--burnin", type=int, default=0, help="drop the samples up to this generation")
    a = ap.parse_args(argv)
    res = summary(a.path, a.burnin)
    print("statistic", "p(rep<=obs)", "observed_mean", "replicate_mean", "replicates", sep="\t")
    for name, r in res.items():
        print(name, "%.6g" % r["p"], "%.17g" % r["observed_mean"], "%.17g" % r["replicate_mean"], r["replicates"],
              sep="\t")


if __name__ == "__main__":
    main(sys.argv[1:])
