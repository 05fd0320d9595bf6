"""What one posterior predictive replicate costs (ppc.Replicates.draw), on C1 (narrow.phy, F81 + Gamma-4, the state
recorded for it in tests/golden) and on the C4 shape (1024 taxa x 1M binary columns, GTR + Gamma-4, built as bench.py
builds it; the replicate context holds all 1M columns, uncompressed).

Per replicate, median over --reps replicates (each a new replicate id):
  simulate  device ms of cb_simulate without the download (CUDA events on the engine's stream; the upload of the edge
            list is inside the window), and its bytes -- codes read (every cell) + codes written (every state cell) --
            over the copy bandwidth bench.py uses; the internal-node scratch traffic, when the states do not fit shared
            memory, is printed beside it, computed, not measured;
  lnL       device ms of the replicate's likelihood-only cb_eval (cb_last_eval_ms);
  T         host wall ms of the download (cb_simulate with the download, minus its device ms) plus the pattern
            compression of the replicate and the statistic;
  total     host wall ms of Replicates.draw (P matrices, simulate, lnL, download, T).
Prints the card and its power limit first.

    python profiles/microbench/ppc_cost.py [--reps 5] [--patterns 1000000] [--skip-c4]
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
sys.path.insert(0, os.path.join(REPO, "oracle"))


def card():
    try:
        return subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


def measure(label, reps, state, model, n, hbm_gbs):
    from cybayes_b200.ppc import column_weights, multinomial_statistic
    eng = reps.engine
    held = reps._tables(state, model)        # keeps the slot block of these P matrices alive
    _, pi, root, (par, ch, ps), (plan, ps_eval) = held
    S, cb = eng.n_states, np.dtype(eng.code_dtype).itemsize
    n_cells = eng.n_taxa * eng.n_patterns
    reps.draw(state, model, 1, 0)            # warm-up: every allocation, the scratch, both compressions
    rows = {"simulate device ms": [], "lnL device ms": [], "T ms (download + compression)": [], "total wall ms": []}
    state_cells = None
    for r in range(1, n + 1):
        eng.sync()
        eng.mark(0)
        eng.simulate(par, ch, ps, pi, root, 1, r, download=False)
        eng.mark(1)
        eng.sync()
        sim = eng.mark_elapsed_ms()
        eng.eval(None, plan.nodes, plan.children, ps_eval, pi, want_snapshot=False)
        lnl = eng.last_eval_ms()
        t0 = time.perf_counter()
        codes = eng.simulate(par, ch, ps, pi, root, 1, r)
        t1 = time.perf_counter()
        multinomial_statistic(column_weights(codes))
        t2 = time.perf_counter()
        state_cells = int(np.count_nonzero(codes < S))
        t3 = time.perf_counter()
        reps.draw(state, model, 1, r)
        t4 = time.perf_counter()
        rows["simulate device ms"].append(sim)
        rows["lnL device ms"].append(lnl)
        rows["T ms (download + compression)"].append(max(0.0, (t1 - t0) * 1e3 - sim) + (t2 - t1) * 1e3)
        rows["total wall ms"].append((t4 - t3) * 1e3)
    moved = (n_cells + state_cells) * cb
    sim_ms = statistics.median(rows["simulate device ms"])
    print(f"--- {label}: {eng.n_taxa} taxa x {eng.n_patterns} columns, S = {S}, C = {eng.n_cats}, {cb}-byte codes")
    for k, v in rows.items():
        print(f"{k:34s} median {statistics.median(v):10.3f}   [{min(v):.3f}, {max(v):.3f}]")
    print(f"simulate bytes (codes read + written): {moved / 1e9:.3f} GB -> {moved / (sim_ms * 1e-3) / 1e9:.0f} GB/s "
          f"= {moved / (sim_ms * 1e-3) / 1e9 / hbm_gbs:.2f} of {hbm_gbs:.0f} GB/s")
    if (eng.n_taxa - 1) * 128 * cb > 96 * 1024:
        scratch = (eng.n_taxa - 1) * eng.n_patterns * cb
        print(f"internal states in the global scratch (computed, not measured): {scratch / 1e9:.3f} GB written, "
              f"{2 * scratch / 1e9:.3f} GB read")
    del held


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--taxa", type=int, default=1024)
    ap.add_argument("--patterns", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-c4", action="store_true")
    a = ap.parse_args()
    print("card:", card(), flush=True)
    import golden_io
    from cybayes_b200 import config, likelihood
    from cybayes_b200.alignment import LeafMatrices
    from cybayes_b200.driver import load_alignment
    from cybayes_b200.ppc import Replicates
    from cybayes_b200.synthetic import SyntheticAlignment
    from bench import measured_peaks
    hbm_gbs, src = measured_peaks()
    print(f"copy bandwidth: {hbm_gbs:.0f} GB/s, {src}", flush=True)

    case = golden_io.load_cases()["narrow_F81"]
    load_alignment(golden_io.data_path(case), case["dtype"], case["reader"])
    config.MODEL, config.NORM_BETA = case["model"], case["norm_beta"]
    tree, pi, rates, _, _ = golden_io.case_state(case)
    state = {"tree": tree, "root": case["root"], "pi": pi, "rates": rates, "srates": 0.8, "logLikehood": 0.0}
    reps = Replicates(config.LEAF_LLMAT, config.N_CATS)
    measure("C1 narrow.phy F81", reps, state, "F81", a.reps, hbm_gbs)
    reps.close()
    likelihood.reset_engines()
    if a.skip_c4:
        return
    N, P, S = a.taxa, a.patterns, 2
    aln = SyntheticAlignment(N, P, S, 20260101, block_sites=125000)   # bench.py's SEED and BLOCK
    codes = aln.codes(0, P)
    config.N_TAXA, config.N_CHARS, config.N_SITES, config.MODEL, config.IN_DTYPE, config.N_CATS = N, S, P, "GTR", "bin", 4
    leaves = LeafMatrices(codes, S, np.ones((1, S)))
    reps = Replicates(leaves, 4)
    state = {"tree": aln.tree, "root": aln.root, "pi": aln.pi, "rates": aln.er, "srates": 0.5, "logLikehood": 0.0}
    measure("C4 shape", reps, state, "GTR", a.reps, hbm_gbs)
    reps.close()


if __name__ == "__main__":
    main()
