#!/usr/bin/env python3
"""Generate the golden fixtures under tests/golden/ from the UNMODIFIED reference.

TEST INFRASTRUCTURE.  Runs only in the build container (needs /root/reference for
the data files and oracle/_ref/ for the compiled reference, see oracle/build_ref.sh).
The GPU box never runs this; it reads the committed fixtures.

What is pinned (the reference ships no tests of its own, SURVEY.md section 4):

* ``cases.json``  -- for every (dataset, reader, model) case: the reader outputs
  (alphabet, taxa, digest of the leaf 0/1 matrices, utils.pyx:94-120), the
  start state produced by ``state_init`` with the driver's seeding
  (mat_mcmc_gamma.py:7-8,46; mcmc_gamma.pyx:573-593): pi, rates, tree dict in
  insertion order, root, srates, postorder, site rates, NORM_BETA, a sample of
  P(t) matrices, the initial lnL of ``ML_gamma.matML`` (ML_gamma.pyx:7-42), per
  node checksums of the cached partials, and a handful of dirty-path
  ``cache_matML`` evaluations (ML_gamma.pyx:83-118) on that state.
* ``traces/<case>.tsv`` -- the per-generation stdout of the unmodified driver run
  with ``-t 1`` (iter, current lnL, proposed lnL, tree length, param, move) plus
  the ``.log`` columns (lnL, TL, alpha) and the final accept/total counters.
"""
import hashlib
import io
import json
import os
import random
import subprocess
import sys
import contextlib

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REF_BUILD = os.path.join(REPO, "oracle", "_ref")
REF_DATA = "/root/reference/data"
DATA_OUT = os.path.join(HERE, "data")

# (case name, data file, reader, model, dtype flag, n_gen for the trace or 0)
CASES = [
    ("binary_F81", "binary.phy", "readBinaryPhy", "F81", "bin", 300),
    ("twoStates_F81", "twoStates.phy", "readBinaryPhy", "F81", "bin", 300),
    ("twoStates_JC", "twoStates.phy", "readBinaryPhy", "JC", "bin", 300),
    ("narrow_F81", "narrow.phy", "readBinaryPhy", "F81", "bin", 3000),
    ("narrow_JC", "narrow.phy", "readBinaryPhy", "JC", "bin", 500),
    ("narrow_GTR", "narrow.phy", "readBinaryPhy", "GTR", "bin", 0),
    ("broad_F81", "broad.phy", "readBinaryPhy", "F81", "bin", 300),
    ("phon_ringe_JC", "phon_ringe.phy", "readMultiPhy", "JC", "multi", 500),
    ("phon_ringe_F81", "phon_ringe.phy", "readMultiPhy", "F81", "multi", 500),
    ("phon_ringe_GTR", "phon_ringe.phy", "readMultiPhy", "GTR", "multi", 300),
    ("ie42_JC", "data-ie-42-208_prog.phy", "readMultiPhy", "JC", "multi", 200),
    ("ie42_GTR", "data-ie-42-208_prog.phy", "readMultiPhy", "GTR", "multi", 60),
    ("ielex2016_JC", "IELex-2016.prog.phy", "readPhy", "JC", "multi", 0),
    ("ielex_multistate_F81", "ielex_multistate.phy", "readPhy", "F81", "multi", 0),
    ("german_multistate_JC", "German_multistate.phy", "readPhy", "JC", "multi", 0),
]


def _leaf_digest(ll_mats, n_taxa):
    import numpy as np
    h = hashlib.sha256()
    for k in range(1, n_taxa + 1):
        m = np.ascontiguousarray(ll_mats[k])
        assert set(np.unique(m)).issubset({0.0, 1.0})
        h.update(np.packbits(m.astype(bool), axis=None).tobytes())
    return h.hexdigest()


def case_vectors(name, fname, reader, model, dtype):
    """Runs in a fresh interpreter (see main) with oracle/_ref on sys.path."""
    import numpy as np
    import config, utils, mcmc_gamma, ML_gamma  # the compiled reference

    np.random.seed(1234)
    random.seed(1234)
    path = os.path.join(REF_DATA, fname)
    with contextlib.redirect_stdout(io.StringIO()):  # readPhy prints every row
        (config.N_TAXA, config.N_CHARS, config.ALPHABET, site_dict, config.LEAF_LLMAT,
         config.TAXA, config.N_SITES) = getattr(utils, reader)(path)
    config.IN_DTYPE, config.MODEL = dtype, model
    config.N_NODES = 2 * config.N_TAXA - 1
    if model == "JC":
        config.NORM_BETA = config.N_CHARS / (config.N_CHARS - 1)
    st = mcmc_gamma.state_init()
    site_rates = mcmc_gamma.get_siterates(st["srates"])
    lnl, cache = ML_gamma.matML(st["pi"], st["root"], config.LEAF_LLMAT, st["postorder"],
                                st["transitionMat"], config.N_SITES, config.N_TAXA, config.N_CATS)
    pi = np.asarray(st["pi"]).tolist()
    rates = np.asarray(st["rates"]).tolist()
    tree = [[int(p), int(c), float(t)] for (p, c), t in st["tree"].items()]
    out = {
        "name": name, "file": fname, "reader": reader, "model": model, "dtype": dtype,
        "n_taxa": int(config.N_TAXA), "n_chars": int(config.N_CHARS), "n_sites": int(config.N_SITES),
        "alphabet": list(config.ALPHABET), "taxa": list(config.TAXA),
        "leaf_digest": _leaf_digest(config.LEAF_LLMAT, config.N_TAXA),
        "pi": pi, "rates": rates if len(rates) <= 300 else None,
        "rates_digest": hashlib.sha256(np.asarray(st["rates"]).tobytes()).hexdigest(),
        "tree": tree, "root": int(st["root"]), "srates": float(st["srates"]),
        "postorder": [[int(p), int(c)] for p, c in st["postorder"]],
        "site_rates": [float(x) for x in site_rates],
        "norm_beta": float(config.NORM_BETA),
        "lnL": float(lnl),
    }
    # sample of P(t) matrices: first, middle and last edge (dict order) x all categories
    keys = list(st["tree"].keys())
    sample = [keys[0], keys[len(keys) // 2], keys[-1]]
    pm = {}
    for (p, c) in sample:
        mats = [np.asarray(st["transitionMat"][k][p, c]) for k in range(config.N_CATS)]
        if config.N_CHARS <= 8:
            pm[f"{p},{c}"] = [m.tolist() for m in mats]
        else:  # store row 0, the diagonal and the row sums only
            pm[f"{p},{c}"] = [{"row0": m[0].tolist(), "diag": np.diag(m).tolist(),
                               "rowsum": m.sum(axis=1).tolist()} for m in mats]
    out["pmat_sample"] = pm
    # per-node checksums of the cached partials (sum over states and sites, per category)
    chk = {}
    for node in sorted(cache[0].keys()):
        chk[str(node)] = [float(np.sum(cache[k][node])) for k in range(config.N_CATS)]
    out["partial_sums"] = chk
    if config.N_TAXA <= 10:
        out["partials"] = {str(n): [np.asarray(cache[k][n]).tolist() for k in range(config.N_CATS)]
                           for n in sorted(cache[0].keys())}
    # dirty-path evaluations: scale one edge by 1.7 (F81/JC/GTR via get_edge_transition_mat)
    rev = mcmc_gamma.adjlist2reverse_nodes_dict(st["tree"])
    dirty = []
    rng = random.Random(99)
    for (p, c) in rng.sample(keys, min(6, len(keys))):
        new_t = st["tree"][p, c] * 1.7
        saved = [st["transitionMat"][k][p, c] for k in range(config.N_CATS)]
        for k, r in enumerate(site_rates):
            st["transitionMat"][k][p, c] = mcmc_gamma.get_edge_transition_mat(st["pi"], st["rates"], new_t * r)
        path2root = mcmc_gamma.get_path2root(rev, c, st["root"])
        l2, _ = ML_gamma.cache_matML(st["pi"], st["root"], config.LEAF_LLMAT, cache, path2root,
                                     st["postorder"], st["transitionMat"], config.N_SITES,
                                     config.N_TAXA, config.N_CATS)
        for k in range(config.N_CATS):
            st["transitionMat"][k][p, c] = saved[k]
        dirty.append({"edge": [int(p), int(c)], "new_t": float(new_t),
                      "path": [int(x) for x in path2root], "lnL": float(l2)})
    out["dirty"] = dirty
    return out


def run_trace(name, fname, model, dtype, n_gen):
    """Run the byte-compiled, unmodified driver with -t 1 and keep its per-generation output."""
    out_prefix = f"/tmp/golden_{name}"
    cmd = [sys.executable, "mat_mcmc_gamma.code", "-i", os.path.join(REF_DATA, fname), "-m", model,
           "-n", str(n_gen), "-t", "1", "-d", dtype, "-o", out_prefix]
    res = subprocess.run(cmd, cwd=REF_BUILD, capture_output=True, text=True, check=True)
    gens, counters, init_lnl = [], [], None
    for line in res.stdout.splitlines():
        f = line.split("\t")
        if line.startswith("Initial Likelihood"):
            init_lnl = line.split()[-1]
        elif len(f) == 6 and f[0].isdigit():
            gens.append(f)
        elif line.startswith("(np.str_(") or line.startswith("('"):
            counters.append(line)
    logrows = [l.split("\t") for l in open(out_prefix + ".log").read().splitlines()[1:]]
    assert len(gens) == n_gen == len(logrows), (len(gens), n_gen, len(logrows))
    trees = open(out_prefix + ".trees").read()
    os.makedirs(os.path.join(HERE, "traces"), exist_ok=True)
    with open(os.path.join(HERE, "traces", name + ".tsv"), "w") as fh:
        fh.write(f"# unmodified reference driver, seed 1234, -n {n_gen} -t 1; init_lnL={init_lnl}\n")
        fh.write(f"# trees_sha256={hashlib.sha256(trees.encode()).hexdigest()}\n")
        fh.write("# last_tree=" + trees.strip().splitlines()[-1].split("\t")[1] + "\n")
        for c in counters:
            fh.write("# counter " + c + "\n")
        fh.write("iter\tcurrent_ll\tproposed_ll\tTL\tparam\tmove\tstate_lnL\tlog_TL\talpha\n")
        for g, lr in zip(gens, logrows):
            assert g[0] == lr[0]
            fh.write("\t".join(g + lr[1:]) + "\n")


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "--case":
        sys.path.insert(0, REF_BUILD)
        idx = int(sys.argv[2])
        print("@@JSON@@" + json.dumps(case_vectors(*CASES[idx][:5])))
        return
    os.makedirs(DATA_OUT, exist_ok=True)
    cases = []
    for i, (name, fname, reader, model, dtype, n_gen) in enumerate(CASES):
        # input alignments are fixtures (data, not code): keep a copy beside the goldens
        dst = os.path.join(DATA_OUT, fname)
        if not os.path.exists(dst):
            with open(os.path.join(REF_DATA, fname), "rb") as s, open(dst, "wb") as d:
                d.write(s.read())
        res = subprocess.run([sys.executable, __file__, "--case", str(i)], capture_output=True,
                             text=True, check=True)
        payload = [l for l in res.stdout.splitlines() if l.startswith("@@JSON@@")][0]
        case = json.loads(payload[len("@@JSON@@"):])
        case["trace_gens"] = n_gen
        cases.append(case)
        print(f"{name}: lnL={case['lnL']!r}", flush=True)
        if n_gen and reader != "readPhy":
            run_trace(name, fname, model, dtype, n_gen)
    with open(os.path.join(HERE, "cases.json"), "w") as fh:
        json.dump({"generator": "tests/golden/make_golden.py", "cases": cases}, fh, indent=0)


if __name__ == "__main__" and not (len(sys.argv) > 1 and sys.argv[1] in ("--nongamma", "--c1-100k", "--random-inputs")):
    main()


# ---- non-Gamma driver (mat_mcmc.py + mcmc.pyx + ML.pyx): traces only -------------------------------
NONGAMMA = [("ng_binary_F81", "binary.phy", "F81", "bin", 300), ("ng_phon_ringe_JC", "phon_ringe.phy", "JC", "multi", 300),
            ("ng_narrow_F81", "narrow.phy", "F81", "bin", 400)]


def run_trace_nongamma(name, fname, model, dtype, n_gen):
    out_prefix = f"/tmp/golden_{name}"
    cmd = [sys.executable, "mat_mcmc.code", "-i", os.path.join(REF_DATA, fname), "-m", model, "-n", str(n_gen),
           "-t", "1", "-d", dtype, "-o", out_prefix]
    res = subprocess.run(cmd, cwd=REF_BUILD, capture_output=True, text=True, check=True)
    gens = [l.split("\t") for l in res.stdout.splitlines() if len(l.split("\t")) == 6 and l.split("\t")[0].isdigit()]
    init = [l for l in res.stdout.splitlines() if l.startswith("Initial Likelihood")][0].split()[-1]
    assert len(gens) == n_gen
    with open(os.path.join(HERE, "traces", name + ".tsv"), "w") as fh:
        fh.write(f"# unmodified reference driver mat_mcmc.py, seed 1234, -n {n_gen} -t 1; init_lnL={init}\n")
        fh.write("iter\tstate_lnL\tproposed_ll\tTL\tparam\tmove\n")
        for g in gens:
            fh.write("\t".join(g) + "\n")


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "--nongamma":
    for args in NONGAMMA:
        run_trace_nongamma(*args)
        print("trace", args[0])


# ---- C1 at its stated length (README.md:46): narrow.phy F81, -n 100000 -t 1000 -------------------------------
C1_MOVES = ["scale_edge", "node_slider", "rooted_NNI", "externalSPR", "mvDualSlider", "scale_alpha"]


def run_c1_100k(n_gen=100000, thin=1000, workdir="/tmp"):
    """Two runs of the unmodified driver on data/narrow.phy (seed 1234): the README command itself
    (`-n 100000 -t 1000`: its .log is kept verbatim, its .trees as digest + last tree, plus the counters) and the
    same chain with `-t 1`, from which a compact per-generation record is kept: move id and accept bit for all
    100 000 generations, the proposed lnL of every 100th.  Existing outputs in `workdir` are reused."""
    import numpy as np
    runs = {}
    for t in (thin, 1):
        prefix = os.path.join(workdir, f"c1_t{t}")
        if not (os.path.exists(prefix + ".log") and os.path.exists(prefix + ".stdout")):
            cmd = [sys.executable, "mat_mcmc_gamma.code", "-i", os.path.join(REF_DATA, "narrow.phy"), "-m", "F81",
                   "-n", str(n_gen), "-t", str(t), "-d", "bin", "-o", prefix]
            with open(prefix + ".stdout", "w") as fh:
                subprocess.run(cmd, cwd=REF_BUILD, stdout=fh, check=True)
        runs[t] = prefix
    out_dir = os.path.join(HERE, "traces")
    # (a) the README run
    p = runs[thin]
    log = open(p + ".log").read()
    trees = open(p + ".trees").read()
    stdout = open(p + ".stdout").read().splitlines()
    counters = [l for l in stdout if l.startswith("(np.str_(") or l.startswith("('")]
    init = [l for l in stdout if l.startswith("Initial Likelihood")][0].split()[-1]
    assert len(log.splitlines()) == n_gen // thin + 1
    with open(os.path.join(out_dir, "c1_narrow_F81_100k.log"), "w") as fh:
        fh.write(log)
    meta = {"cmd": f"mat_mcmc_gamma.py -i data/narrow.phy -m F81 -n {n_gen} -t {thin} -d bin (seed 1234, unmodified reference)",
            "init_lnL": init, "counters": counters, "trees_sha256": hashlib.sha256(trees.encode()).hexdigest(),
            "last_tree": trees.strip().splitlines()[-1].split("\t")[1], "moves": C1_MOVES}
    # (b) the same chain, every generation
    p = runs[1]
    gens = [l.split("\t") for l in open(p + ".stdout").read().splitlines()
            if len(l.split("\t")) == 6 and l.split("\t")[0].isdigit()]
    logrows = [l.split("\t") for l in open(p + ".log").read().splitlines()[1:]]
    assert len(gens) == n_gen == len(logrows)
    # both runs are one chain: the thinned .log rows are rows of the -t 1 .log
    thinned = [l.split("\t") for l in log.splitlines()[1:]]
    for row in thinned:
        assert logrows[int(row[0]) - 1] == row, row
    move = np.array([C1_MOVES.index(g[5]) for g in gens], dtype=np.uint8)
    accepted = np.array([lr[1] == g[2] for g, lr in zip(gens, logrows)], dtype=bool)
    every = 100
    sampled = np.array([float(g[2]) for g in gens[every - 1::every]])
    np.savez_compressed(os.path.join(out_dir, "c1_narrow_F81_100k.npz"), move=move, accepted=np.packbits(accepted),
                        proposed_ll_every_100=sampled)
    meta["accepted_total"] = int(accepted.sum())
    with open(os.path.join(out_dir, "c1_narrow_F81_100k.json"), "w") as fh:
        json.dump(meta, fh, indent=0)
    print("c1 100k:", meta["accepted_total"], "accepted;", counters)


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "--c1-100k":
    run_c1_100k()


# ---- seeded random inputs of tests/test_oracle.py: their expected outputs, stored ---------------------------------
def random_input_vectors(out, source):
    """Write golden_io.random_vectors of every golden_io.random_inputs case to `out` (.npz), computed by the compiled
    reference (source "reference": oracle/_ref; run this in a fresh interpreter, its module names are top-level) or by
    the NumPy oracle (source "oracle"), with a `source` entry naming which."""
    import numpy as np
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import golden_io
    import pruning_oracle as oracle
    if source == "reference":
        sys.path.insert(0, REF_BUILD)
        import config, mcmc_gamma, ML_gamma  # the compiled reference
    rec = {"source": np.array(source)}
    for i, c in enumerate(golden_io.random_inputs()):
        tree, root, pi, ll, N, P = c["tree"], c["root"], c["pi"], c["ll"], c["n_taxa"], c["n_sites"]
        if source == "reference":
            config.N_TAXA, config.N_CHARS, config.N_SITES, config.MODEL, config.IN_DTYPE = N, c["S"], P, c["model"], c["dtype"]
            config.NORM_BETA = c["beta"]
            edges = mcmc_gamma.postorder(mcmc_gamma.adjlist2nodes_dict(tree), root)[::-1]
            rates = mcmc_gamma.get_siterates(0.8)
            tm = [mcmc_gamma.get_prob_t(pi, tree, c["er"], r) for r in rates]
            lnl, cache = ML_gamma.matML(pi, root, ll, edges, tm, P, N, 4)
            path = mcmc_gamma.get_path2root(mcmc_gamma.adjlist2reverse_nodes_dict(tree), 3, root)
            l2, _ = ML_gamma.cache_matML(pi, root, ll, cache, path, edges, tm, P, N, 4)
        else:
            edges = oracle.edge_order(tree, root, N)
            rates = oracle.site_rates(0.8)
            tm = [oracle.prob_t(c["model"], c["dtype"] == "bin", pi, tree, c["er"], r, beta=c["beta"]) for r in rates]
            lnl, cache = oracle.mat_ml(pi, root, ll, edges, tm, P, N)
            path = oracle.path_to_root(oracle.parent_of(tree), 3, root)
            l2, _ = oracle.cache_mat_ml(pi, root, ll, cache, path, edges, tm, P, N)
        rec.update(golden_io.random_vectors(i, c, edges, rates, tm, lnl, path, l2))
    np.savez(out, **rec)


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "--random-inputs":
    # python tests/golden/make_golden.py --random-inputs [OUT] [reference|oracle]
    random_input_vectors(sys.argv[2] if len(sys.argv) > 2 else os.path.join(HERE, "random_inputs.npz"),
                         sys.argv[3] if len(sys.argv) > 3 else "reference")
