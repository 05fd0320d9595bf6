"""What per-site output costs on the C4 shape (1024 taxa x 1M binary patterns, GTR + Gamma-4, built as bench.py builds
it): cb_eval against cb_eval_sites for a full pass (alternating, same operands), and a root-only cb_eval_sites against
a kept snapshot, with and without the rate-category posteriors.

Device time: CUDA events on the engine's stream around each call (the D2H copy of the per-site arrays included); host
wall time: perf_counter around the call, which returns after the copy.  Prints the card and its power limit first.

    python profiles/microbench/site_lnl_cost.py [--reps 10] [--patterns 1000000]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)


def card():
    try:
        return subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--taxa", type=int, default=1024)
    ap.add_argument("--patterns", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    print("card:", card(), flush=True)
    from cybayes_b200 import _lib, config, likelihood
    from cybayes_b200.alignment import LeafMatrices
    from cybayes_b200.subst import gtr_eigensystem
    from cybayes_b200.synthetic import SyntheticAlignment

    N, P, C, S = a.taxa, a.patterns, 4, 2
    aln = SyntheticAlignment(N, P, S, 20260101, block_sites=125000)   # bench.py's SEED and BLOCK
    codes = aln.codes(0, P)
    config.N_TAXA, config.N_CHARS, config.N_SITES, config.MODEL, config.IN_DTYPE = N, S, P, "GTR", "bin"
    leaves = LeafMatrices(codes, S, np.ones((1, S)))
    eng, _ = likelihood.engine_for(leaves, C)
    plan = likelihood._plan_for(aln.edge_order())
    ekeys = list(aln.tree.keys())
    block = eng.alloc_slots(len(ekeys) * C)
    slots = np.arange(block.base, block.base + block.n, dtype=np.int32)
    d = np.array([aln.tree[e] * r for r in aln.rates for e in ekeys])
    eng.queue_build(_lib.CB_MODEL_GTR_EIG, aln.pi, 0.0, gtr_eigensystem(aln.pi, aln.er), slots, d)
    slot_of = {(k, e): block.base + k * len(ekeys) + i for k in range(C) for i, e in enumerate(ekeys)}
    pslots = np.array([[slot_of[k, e] for k in range(C)] for e in plan.edge_keys], dtype=np.int32)
    pi, root, kids = aln.pi, aln.root, plan.kids
    r_nodes, r_children = np.array([root], dtype=np.int32), np.array(kids[root], dtype=np.int32)
    r_pslots = np.array([[slot_of[k, (root, c)] for k in range(C)] for c in kids[root]], dtype=np.int32)
    print(f"engine: {eng.n_patterns} patterns of {P} columns, {len(plan.nodes)} ops", flush=True)

    def timed(fn):
        eng.sync()
        eng.mark(0)
        t0 = time.perf_counter()
        out = fn()
        wall = (time.perf_counter() - t0) * 1e3
        eng.mark(1)
        eng.sync()
        return eng.mark_elapsed_ms(), wall, out

    full_eval = lambda: eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=False)[0]   # noqa: E731
    full_sites = lambda: eng.eval_sites(None, plan.nodes, plan.children, pslots, pi, categories=True)[0]  # noqa: E731
    full_sites_l = lambda: eng.eval_sites(None, plan.nodes, plan.children, pslots, pi)[0]  # noqa: E731
    _, snap = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True)
    root_l = lambda: eng.eval_sites(snap, r_nodes, r_children, r_pslots, pi)[0]  # noqa: E731
    root_q = lambda: eng.eval_sites(snap, r_nodes, r_children, r_pslots, pi, categories=True)[0]  # noqa: E731
    root_eval = lambda: eng.eval(snap, r_nodes, r_children, r_pslots, pi, want_snapshot=False)[0]  # noqa: E731
    arms = {"full cb_eval": full_eval, "full cb_eval_sites (l)": full_sites_l, "full cb_eval_sites (l + q)": full_sites,
            "root-only cb_eval": root_eval, "root-only cb_eval_sites (l)": root_l,
            "root-only cb_eval_sites (l + q)": root_q}
    for fn in arms.values():   # warm-up: every shape, every allocation
        fn()
        fn()
    res = {k: ([], []) for k in arms}
    lnls = {k: set() for k in arms}
    for _ in range(a.reps):    # alternate the arms so that drift hits all of them alike
        for k, fn in arms.items():
            dev, wall, lnl = timed(fn)
            res[k][0].append(dev)
            res[k][1].append(wall)
            lnls[k].add(lnl)
    assert len(set().union(*lnls.values())) == 1, lnls   # every arm computes the same lnL, bit for bit
    Pp = -(-eng.n_patterns // 64) * 64   # what the kernels see: the compressed, padded pattern count
    print(f"computed, not measured: per-site outputs (l + q) (1 + C) * 8 * P = {(1 + C) * 8 * Pp / 1e6:.1f} MB; a root-only "
          f"op reads two child partials of 2 * C * 8 * P + 4 * P bytes = 2 x {(2 * C * 8 + 4) * Pp / 1e6:.1f} MB")
    print(f"{'arm':34s} {'device ms median [min, max]':>30s} {'host wall ms median':>20s}")
    for k, (dev, wall) in res.items():
        print(f"{k:34s} {statistics.median(dev):10.3f} [{min(dev):.3f}, {max(dev):.3f}] {statistics.median(wall):14.3f}")
    eng.release_snapshot(snap)


if __name__ == "__main__":
    main()
