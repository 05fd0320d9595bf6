#!/usr/bin/env python3
"""Benchmark of the tree-likelihood hot path (contract in the task statement / DESIGN.md section 5).

  python bench.py [--gpus N --steps K --warmup W]            our arm (CUDA engine), config C4
  python bench.py --impl reference [...]                      the reference's own CPU path, same config
  python bench.py --config C5|C1|C2|C3 [...]                  the other BASELINE.json configurations, same schema
  python bench.py --dump-outputs DIR [...]                    also write the last timed step's outputs to DIR

Workload at the defaults (BASELINE.json, config C4): synthetic 1024 taxa x 1,000,000 binary site patterns,
GTR + discrete-Gamma-4, one *step* = one full Felsenstein pruning pass (log-likelihood evaluation) keeping the
partial cache.  For N > 1 the patterns are sharded over the ranks (one process per GPU, torchrun), each rank runs
the same op list on its slice and the only exchange is the scalar NCCL all-reduce inside the library: strong
scaling, `value` = whole-alignment evals/s.

One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

os.environ.setdefault("CYBAYES_COMPRESS_MAX_SITES", "0")  # patterns are used as generated (weights 1)
REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

import numpy as np  # noqa: E402

SEED = 20260101
BLOCK = 125000          # generation / sharding granule: 1M = 8 blocks
METRIC = "tree log-likelihood evals/sec"
UNIT = "evals/s"
DATA = os.path.join(REPO, "tests", "golden", "data")
REAL = {   # BASELINE.json configs[0..2]
    "C1": ("narrow.phy", "readBinaryPhy", "bin", "F81"),
    "C2": ("IELex-2016.prog.phy", "readPhy", "multi", "JC"),
    "C3": ("ielex_multistate.phy", "readPhy", "multi", "F81"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps: likelihood evaluations for C4 / C5 (default 20), MCMC generations for C1 - C3 "
                         "(default 20000 / 4000 / 4000)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C4", choices=["C4", "C5", "C1", "C2", "C3"])
    ap.add_argument("--taxa", type=int, default=None)
    ap.add_argument("--patterns", type=int, default=None)
    ap.add_argument("--ref-chunk", type=int, default=12500, help="sites per matML call of --impl reference (divides 125000)")
    ap.add_argument("--no-extras", action="store_true", help="skip cpu_baseline / dirty-path / MCMC extras")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy, float64. C4 / C5: "
                         "lnL.npy and partial_log.npy, the natural log of a fixed, seeded sample of the kept partial "
                         "cache; C5 on one GPU at the default size keeps no cache and writes lnL.npy only, and with "
                         "--gpus > 1 the sample is drawn from rank 0's patterns, so compare runs with equal --gpus. "
                         "C1 - C3: the final state of the chain (lnL, pi, rates, alpha, tree)")
    a = ap.parse_args()
    if a.steps is not None and a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.steps is None and a.config not in REAL:
        a.steps = 20
    if a.dump_outputs is not None and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if a.taxa is None:
        a.taxa = 512 if a.config == "C5" else 1024
    if a.patterns is None:
        a.patterns = 200000 if a.config == "C5" else 1000000
    a.warmup = max(a.warmup, 3)
    return a


def workload_name(a):
    if a.config == "C5":
        return (f"C5: synthetic {a.taxa} taxa x {a.patterns} site patterns x 64 states, GTR + Gamma-4, full pruning "
                "pass (likelihood evaluation)")
    return (f"C4: synthetic {a.taxa} taxa x {a.patterns} binary site patterns, GTR + Gamma-4, "
            "full pruning pass (likelihood evaluation) with the partial cache kept")


def config_dict(a):
    """The same dict for both arms (`--impl ours` / `--impl reference`)."""
    S = 64 if a.config == "C5" else 2
    per_gpu = -(-a.patterns // a.gpus)
    return {"workload": workload_name(a), "n_taxa": a.taxa, "n_patterns": a.patterns, "n_states": S, "n_cats": 4,
            "model": "GTR", "parallelism": f"site-sharded x{a.gpus}", "patterns_per_gpu": per_gpu,
            "l2": "inputs per step (GBs of partials per GPU) are far larger than the 126 MB L2; no flush"}


def measured_peaks():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


_NVML_SAMPLER = r"""
import os, sys, time
import pynvml as nv
nv.nvmlInit()
h = nv.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
out = open(sys.argv[2], "w")
print("ready", mx, file=out, flush=True)
parent, t_max = os.getppid(), time.time() + 1800
while os.getppid() == parent and time.time() < t_max:   # never outlives the bench process
    t = time.time()
    print(t, nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), int(reasons(h)), file=out, flush=True)
    time.sleep(0.005)
"""


class ClockSampler:
    """SM clock and throttle reasons of one GPU while the timed region runs.  A helper process polls NVML every few
    milliseconds with wall-clock stamps (the timed region of a sharded run is only tens of milliseconds long: a
    100 ms `nvidia-smi -lms` loop can miss it entirely); it is started before the warm-up steps, `begin()` / `stop()`
    bracket the timed region and only the samples in between are reported.  Without pynvml: `nvidia-smi -lms`."""
    SMI_FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                  "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    # NVML reason bits (nvml.h): SwPowerCap 0x4, HwSlowdown 0x8, SwThermalSlowdown 0x20, HwThermalSlowdown 0x40
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, device):
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.tmp.close()
        self.t_begin = self.t_end = None
        self.mode, self.proc = "nvml", None
        try:
            import pynvml  # noqa: F401  (only to choose the sampler; the polling happens in the helper process)
            self.proc = subprocess.Popen([sys.executable, "-c", _NVML_SAMPLER, str(device), self.tmp.name],
                                         stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            for _ in range(400):   # wait until the helper has initialised NVML (first line of its file)
                if os.path.getsize(self.tmp.name) > 0 or self.proc.poll() is not None:
                    break
                time.sleep(0.005)
            if self.proc.poll() is not None or os.path.getsize(self.tmp.name) == 0:
                raise RuntimeError("NVML sampler did not start")
        except Exception:
            self._kill()
            self.mode = "smi"
            try:
                self.proc = subprocess.Popen(["nvidia-smi", "-i", str(device), f"--query-gpu={self.SMI_FIELDS}",
                                              "--format=csv,noheader,nounits", "-lms", "20"],
                                             stdout=open(self.tmp.name, "w"), stderr=subprocess.DEVNULL)
            except Exception:
                self.proc = None

    def _kill(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.terminate()
            self.proc.wait()

    def begin(self):
        self.t_begin = time.time()

    def stop(self):
        self.t_end = time.time()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock sampler available"], "samples": 0}
        time.sleep(0.15)   # the power-cap flag lags the load by tens of milliseconds: keep polling a little longer
        self._kill()
        lines = [l.split() if self.mode == "nvml" else l.strip().split(", ") for l in open(self.tmp.name) if l.strip()]
        os.unlink(self.tmp.name)
        if self.mode == "smi":
            sm = [float(r[0]) for r in lines if r[0].replace(".", "").isdigit()]
            mx = [float(r[1]) for r in lines if r[1].replace(".", "").isdigit()]
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            reasons = sorted({names[i] for r in lines if len(r) >= 6 for i in range(4) if r[2 + i].strip() == "Active"})
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                    "reasons": reasons, "samples": len(sm), "sampler": "nvidia-smi -lms 20 (whole run incl. warm-up)"}
        mx = float(lines[0][1]) if lines and lines[0][0] == "ready" else None
        rows = [(float(r[0]), float(r[1]), int(r[2])) for r in lines[1:] if len(r) == 3]
        t0 = self.t_begin if self.t_begin is not None else 0.0
        inside = [r for r in rows if t0 <= r[0] <= self.t_end]
        scope = "timed region"
        if not inside:   # a region shorter than one polling period: the samples just around it
            inside = [r for r in rows if t0 - 0.02 <= r[0] <= self.t_end + 0.005]
            scope = "timed region +- 20 ms"
        mask = run_mask = 0
        for r in inside:
            mask |= r[2]
        for r in rows:
            run_mask |= r[2]
        names = lambda m: sorted(k for k, bit in self.BITS.items() if m & bit)  # noqa: E731
        return {"sm_mhz": statistics.median([r[1] for r in inside]) if inside else None, "sm_max_mhz": mx,
                "reasons": names(mask | run_mask), "reasons_in_timed_region": names(mask), "samples": len(inside),
                "samples_whole_run": len(rows), "sm_mhz_min": min((r[1] for r in inside), default=None),
                "sampler": f"NVML every 5 ms; clocks: {scope}; reasons: warm-up to 150 ms after the timed region (the "
                           "power-cap flag lags the load)"}


DUMP_NODES = 16
DUMP_PARTIAL_BYTES = 48 << 20


def dump_outputs(out_dir, eng, snap, lnl, nodes):
    """--dump-outputs of C4 / C5: what the timed path handed back in its last step, so that two builds can be compared
    output by output on the same seeded inputs.  lnL.npy holds the log-likelihood (float64, shape (1,)).  When the
    step keeps the partial cache (snap >= 0), a fixed, seeded sample of it is read back through the snapshot and
    written as partial_log.npy (DUMP_NODES internal nodes, C, S, patterns): the natural log of each partial
    likelihood, log(mantissa) + exponent * ln 2, which does not depend on where a build rescales and does not
    underflow near the root.  The patterns are as many of this rank's as fit in DUMP_PARTIAL_BYTES, so the files
    stay below 64 MB in all."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "lnL.npy"), np.array([lnl], dtype=np.float64))
    if snap < 0:
        return
    rng = np.random.default_rng(SEED)
    nodes = np.sort(rng.choice(np.asarray(nodes), size=min(DUMP_NODES, len(nodes)), replace=False))
    C, S, P = eng.n_cats, eng.n_states, eng.n_patterns
    n = min(P, DUMP_PARTIAL_BYTES // (len(nodes) * C * S * 8))
    cols = np.sort(rng.choice(P, size=n, replace=False))
    out = np.empty((len(nodes), C, S, n))
    for i, node in enumerate(nodes):
        m, e = eng.read_partial(snap, int(node), with_scale=True)
        with np.errstate(divide="ignore"):     # a partial of exactly 0 is written as -inf
            out[i] = np.log(m[:, :, cols]) + e[cols] * np.log(2.0)
    np.save(os.path.join(out_dir, "partial_log.npy"), out)


def dump_chain_state(out_dir, st):
    """--dump-outputs of C1 - C3: the state the timed chain ends in, float64: lnL.npy (shape (1,)), pi.npy, rates.npy
    (exchangeabilities; empty where the model has none), alpha.npy (shape (1,)) and tree.npy, one row (parent, child,
    branch length) per edge, sorted by (parent, child)."""
    os.makedirs(out_dir, exist_ok=True)
    tree = sorted((p, c, t) for (p, c), t in st["tree"].items())
    rates = np.zeros(0) if st["rates"] is None else st["rates"]
    for name, v in (("lnL", [st["logLikehood"]]), ("pi", st["pi"]), ("rates", rates), ("alpha", [st["srates"]]),
                    ("tree", tree)):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(v, dtype=np.float64))


def host_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


# ------------------------------------------------------------------------------------ reference arm
def reference_available():
    d = os.path.join(REPO, "oracle", "_ref")
    return os.path.exists(d) and any(f.startswith("ML_gamma") and f.endswith(".so") for f in os.listdir(d))


def _ref_setup(taxa, patterns, n_states, seed, block):
    """In a worker process: import the compiled, unmodified reference (oracle/_ref/*.so) and describe the alignment."""
    import random
    sys.path.insert(0, os.path.join(REPO, "oracle", "_ref"))
    import config as rconfig
    import mcmc_gamma as rmcmc
    import ML_gamma as rml
    from cybayes_b200.synthetic import SyntheticAlignment
    aln = SyntheticAlignment(taxa, patterns, n_states, seed, block_sites=block)
    random.seed(1)
    rconfig.N_TAXA, rconfig.N_CHARS = taxa, n_states
    rconfig.MODEL, rconfig.IN_DTYPE = "GTR", ("bin" if n_states == 2 else "multi")
    pi, er = aln.pi.copy(), aln.er.copy()
    tmats = [rmcmc.get_prob_t(pi, aln.tree, er, r) for r in aln.rates]   # the reference's own P(t) (scipy expm)
    return aln, rconfig, rml, tmats, pi


def _ref_leaves(codes, n_states):
    eye = np.eye(n_states)
    return {t + 1: np.ascontiguousarray(eye[codes[t]].T) for t in range(codes.shape[0])}


def _chunk_codes(aln, block, chunk, b, cache):
    """Columns [b * chunk, (b + 1) * chunk) of the alignment (generated in blocks of `block` columns, exactly as the
    GPU arm generates them, so both arms evaluate the same data)."""
    lo = b * chunk
    blk = lo // block
    if cache.get("blk") != blk:
        cache["blk"], cache["codes"] = blk, aln.codes(blk * block, min(aln.n_sites, (blk + 1) * block))
    off = lo - blk * block
    return np.ascontiguousarray(cache["codes"][:, off:off + chunk])


def _ref_worker(rank, n_workers, taxa, patterns, n_states, seed, block, chunk, chunk_ids, n_rounds, barrier, out):
    """One host core of the reference arm: prepares its chunks of the alignment once, then on every barrier
    evaluates all of them with the reference's ML_gamma.matML (ML_gamma.pyx:7-42)."""
    aln, rconfig, rml, tmats, pi = _ref_setup(taxa, patterns, n_states, seed, block)
    edges = aln.edge_order()
    mine, cache = [], {}
    for b in chunk_ids:
        codes = _chunk_codes(aln, block, chunk, b, cache)
        mine.append((_ref_leaves(codes, n_states), codes.shape[1]))
    cache.clear()
    barrier.wait()                       # everybody is prepared
    for _ in range(n_rounds):
        barrier.wait()                   # start of a step
        total = 0.0
        for leaves, n in mine:
            rconfig.N_SITES = n
            lnl, _cache = rml.matML(pi, aln.root, leaves, edges, tmats, n, taxa, 4)
            total += float(lnl)
        out[rank] = total
        barrier.wait()                   # end of a step


def run_reference_arm(a):
    """The reference's own Cython + NumPy matML on every host core.  The reference is single-threaded by
    construction (utils.pyx:3-7) and cannot hold the cache of the full alignment (65 GB at C4), so the alignment is
    cut into site chunks (sites are independent, so the sum of the chunk evaluations IS the reference's evaluation,
    BASELINE.md plan step 3) that are spread over the cores; a step evaluates EVERY chunk once -- the whole
    workload is timed, nothing is extrapolated (unless host memory is too small, which is then stated)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if not reference_available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref is not built (oracle/build_ref.sh)"}))
        return
    import multiprocessing as mp
    S = 64 if a.config == "C5" else 2
    seed = 20260102 if a.config == "C5" else SEED
    block = min(a.patterns, 25000 if a.config == "C5" else BLOCK)     # the generation granule of the GPU arm
    chunk = min(a.ref_chunk if a.config != "C5" else 500, a.patterns)
    if block % chunk:
        raise SystemExit(f"--ref-chunk must divide {block}")
    n_chunks = -(-a.patterns // chunk)
    cores = min(host_cores(), n_chunks)
    leaf_bytes = a.taxa * S * chunk * 8
    cache_bytes = (a.taxa - 1) * 4 * S * chunk * 8
    sampled = False
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 64e9
    ids = list(range(n_chunks))
    # C5 at full size costs ~150 core-seconds per evaluation: bound the step to a sample there (stated below)
    budget_chunks = n_chunks
    if a.config == "C5":
        budget_chunks = min(n_chunks, cores * 2)
    if n_chunks * leaf_bytes + cores * (cache_bytes + leaf_bytes) * 1.5 > 0.8 * avail:
        budget_chunks = min(budget_chunks, cores)
    if budget_chunks < n_chunks:
        ids, sampled = ids[:budget_chunks], True
    per = -(-len(ids) // cores)
    per_worker = [ids[w * per:(w + 1) * per] for w in range(cores)]     # contiguous: a worker generates 1-2 blocks
    ctx = mp.get_context("spawn")
    barrier = ctx.Barrier(cores + 1)
    out = ctx.Array("d", cores)
    n_rounds = a.warmup + a.steps
    procs = [ctx.Process(target=_ref_worker, args=(w, cores, a.taxa, a.patterns, S, seed, block, chunk, per_worker[w],
                                                   n_rounds, barrier, out)) for w in range(cores)]
    for p in procs:
        p.start()
    barrier.wait()
    times, lnl = [], None
    for r in range(n_rounds):
        barrier.wait()
        t0 = time.perf_counter()
        barrier.wait()
        if r >= a.warmup:
            times.append(time.perf_counter() - t0)
        lnl = sum(out[:])
    for p in procs:
        p.join()
    dt = sum(times) / len(times)
    sites = sum(min(chunk, a.patterns - b * chunk) for b in ids)
    value = sites / dt / a.patterns
    if sampled:
        sample = (f"{len(ids)} of {n_chunks} chunks of {chunk} sites on {cores} processes per step ({sites} sites); "
                  f"evals/s of the full {a.patterns}-site alignment extrapolated linearly (sites are independent)")
    else:
        sample = (f"the whole alignment every step: {n_chunks} chunks of {chunk} sites spread over {cores} "
                  "single-threaded processes, nothing extrapolated")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": dt * 1e3 * (a.patterns / sites), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(a),
        "lnL": lnl if not sampled else None, "lnL_sites": sites,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def _cpu_baseline_child(taxa, patterns, n_states, seed, block, chunk, reps, conn):
    """1 core, spawned so the reference's top-level modules never meet the product's: matML on the first chunk."""
    aln, rconfig, rml, tmats, pi = _ref_setup(taxa, patterns, n_states, seed, block)
    codes = _chunk_codes(aln, block, chunk, 0, {})
    leaves = _ref_leaves(codes, n_states)
    edges = aln.edge_order()
    rconfig.N_SITES = codes.shape[1]
    secs, lnl = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        lnl, _cache = rml.matML(pi, aln.root, leaves, edges, tmats, codes.shape[1], taxa, 4)
        secs.append(time.perf_counter() - t0)
        del _cache
    ekeys = list(aln.tree.keys())
    mats = np.stack([np.asarray(tmats[k][e]) for k in range(4) for e in ekeys])
    conn.send((secs, float(lnl), mats))
    conn.close()


def cpu_baseline_chunk(a, n_states, seed, block, chunk, reps=2):
    """The compiled reference on ONE core on chunk 0 of the same alignment.  Returns (dict, lnL of the chunk, the
    reference's own P matrices) -- the GPU is then checked on exactly that chunk with exactly those matrices."""
    if not reference_available():
        return {"value": None, "unit": UNIT, "cores": 1, "kind": "reference",
                "sample": "unavailable: oracle/_ref not built"}, None, None
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    parent, child = ctx.Pipe()
    p = ctx.Process(target=_cpu_baseline_child, args=(a.taxa, a.patterns, n_states, seed, block, chunk, reps, child))
    p.start()
    secs, lnl, mats = parent.recv()
    p.join()
    sec = min(secs)
    n = min(chunk, a.patterns)
    return {"value": 1.0 / (sec * a.patterns / n), "unit": UNIT, "cores": 1, "kind": "reference",
            "sample": f"sites [0, {n}) of {a.patterns}: best of {reps} ML_gamma.matML calls of the compiled reference "
                      f"({sec:.2f} s each), evals/s of the full alignment = linear in the site count (sites are "
                      "independent)"}, lnl, mats


# ------------------------------------------------------------------------------------------ our arm
def _rendezvous(a):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        raise SystemExit(f"--gpus {a.gpus} needs WORLD_SIZE={a.gpus} (launch through torch.distributed.run)")
    dist = None
    if world > 1:
        import torch.distributed as dist  # host-side rendezvous only (gloo); no torch on the device path
        dist.init_process_group("gloo")
    os.environ["CYBAYES_DEVICE"] = str(local)
    return rank, world, local, dist


def _max_over_ranks(dist, *vals):
    if dist is None:
        return vals if len(vals) > 1 else vals[0]
    import torch
    t = torch.tensor(list(vals), dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out = [float(x) for x in t]
    return out if len(out) > 1 else out[0]


def _tables(eng, aln, plan, C):
    """K1: every P(t r) of the tree in one launch; returns (slots, pslots table of the plan, slot_of, ekeys, d)."""
    from cybayes_b200 import _lib
    from cybayes_b200.subst import gtr_eigensystem
    ekeys = list(aln.tree.keys())
    n_e = len(ekeys)
    block = eng.alloc_slots(n_e * C)
    slots = np.arange(block.base, block.base + n_e * C, dtype=np.int32)
    d = np.array([aln.tree[e] * r for r in aln.rates for e in ekeys])
    eng.queue_build(_lib.CB_MODEL_GTR_EIG, aln.pi, 0.0, gtr_eigensystem(aln.pi, aln.er), slots, d)
    slot_of = {(k, e): block.base + k * n_e + i for k in range(C) for i, e in enumerate(ekeys)}
    pslots = np.array([[slot_of[k, e] for k in range(C)] for e in plan.edge_keys], dtype=np.int32)
    return block, slots, pslots, slot_of, ekeys


def run_c4(a):
    rank, world, local, dist = _rendezvous(a)
    from cybayes_b200 import config, likelihood
    from cybayes_b200.alignment import LeafMatrices
    from cybayes_b200.ML_gamma import matML
    from cybayes_b200.synthetic import SyntheticAlignment, shard_bounds

    aln = SyntheticAlignment(a.taxa, a.patterns, 2, SEED, block_sites=BLOCK)
    lo, hi = shard_bounds(a.patterns, rank, world, BLOCK)
    t_gen = time.perf_counter()
    codes = aln.codes(lo, hi)
    t_gen = time.perf_counter() - t_gen
    n_local = codes.shape[1]
    C, S, N = 4, 2, a.taxa

    config.N_TAXA, config.N_CHARS, config.N_SITES, config.MODEL, config.IN_DTYPE = N, S, n_local, "GTR", "bin"
    leaves = LeafMatrices(codes, S, np.ones((1, S)))
    config.LEAF_LLMAT = leaves
    eng, _ = likelihood.engine_for(leaves, C)        # uploads the tips once (resident like model weights)
    if world > 1:
        box = [eng.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        eng.comm_init(box[0], rank, world)

    edges = aln.edge_order()
    plan = likelihood._plan_for(edges)
    block, slots, pslots, slot_of, ekeys = _tables(eng, aln, plan, C)
    n_e = len(ekeys)
    pi = aln.pi

    kept = []

    def step(keep=False):
        lnl, snap = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True)
        if keep:
            kept.append(snap)
        else:
            eng.release_snapshot(snap)
        return lnl

    def barrier():
        if dist is not None:
            dist.barrier()

    clocks = ClockSampler(local) if rank == 0 else None
    for _ in range(a.warmup):
        lnl = step()
    barrier()
    eng.sync()
    if clocks:
        clocks.begin()
    st0 = eng.stats()
    kernel_ms, main_ms = [], []
    eng.host_profile()
    eng.mark(0)
    t0 = time.perf_counter()
    for i in range(a.steps):
        lnl = step(keep=a.dump_outputs is not None and i == a.steps - 1)
        kernel_ms.append(eng.last_eval_ms())
        main_ms.append(eng.last_eval_main_ms())
    eng.mark(1)
    eng.sync()
    wall = time.perf_counter() - t0
    host_prof = eng.host_profile()
    dev_ms = eng.mark_elapsed_ms()
    st1 = eng.stats()
    info = eng.last_eval_info()
    barrier()
    clock_rec = clocks.stop() if clocks else None
    if kept:
        if rank == 0:
            dump_outputs(a.dump_outputs, eng, kept[0], lnl, plan.nodes[:-1])
        eng.release_snapshot(kept[0])
    dev_ms, wall_ms = _max_over_ranks(dist, dev_ms, wall * 1e3)
    ms_per_step = dev_ms / a.steps
    value = 1e3 / ms_per_step

    # Roofline of the dominant kernel (the pruning launch; prune_s2t_kernel<4> from 75 776 patterns per GPU):
    # bytes this evaluation HAS to move, from its op list (stored partials + exponents written once; stored partials
    # read back, tip codes and pattern weights read once; children carried in registers / the shared-memory stack and
    # folded cherries move nothing) / the launch's device time (CUDA events on the launching stream) / measured copy peak.
    k_ms = statistics.mean(main_ms)
    peak, peak_src = measured_peaks()
    required = info["bytes_written"] + info["bytes_read"]
    achieved = required / (k_ms * 1e-3) / 1e9
    alg_bytes = 16.0 * C * S * n_local * (N - 2) + 1.0 * N * n_local + 8.0 * n_local   # SURVEY 8(d): every partial written AND read
    traffic = None
    try:
        with open(os.path.join(REPO, "profiles", "ncu_traffic.json")) as fh:
            tj = json.load(fh)
            if a.patterns == 1000000 and world == 1 and a.taxa == 1024:
                traffic = tj.get("prune_s2t_kernel_dram_bytes_per_eval_1M")
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": "prune_s2t_kernel<4>" if n_local >= 75776 else "prune_s2_kernel<4>",
                "required_bytes_per_eval": required, "bytes_written": info["bytes_written"],
                "bytes_read": info["bytes_read"], "kernel_ms_per_eval": k_ms,
                "eval_ms_incl_prepass": statistics.mean(kernel_ms), "peak_source": peak_src,
                "launches_per_eval": (st1["kernel_launches"] - st0["kernel_launches"]) / a.steps,
                "op_list": {k: info[k] for k in ("ops", "stored", "read_back", "stack_pops", "spills", "cherries_folded",
                                                 "small_records", "launches")},
                "survey_8d": {"algorithmic_bytes_per_eval": alg_bytes, "GBps": alg_bytes / (k_ms * 1e-3) / 1e9,
                              "frac": alg_bytes / (k_ms * 1e-3) / 1e9 / peak,
                              "note": "SURVEY 8(d) counts every non-root partial as written and read back; the walk "
                                      "carries / stacks / folds most of them, so this ratio is not a bandwidth fraction"}}

    # end to end through the reference-facing call: host P matrices (numpy, one dict per category) ->
    # matML -> float.  Timed region holds the H2D of P matrices + op descriptors and the D2H of lnL.
    host_p = eng.download_pmats(slots).reshape(C, n_e, S, S)
    tm_host = [{e: host_p[k, i] for i, e in enumerate(ekeys)} for k in range(C)]
    args = (n_local, N, C)
    for _ in range(3):
        l2, cache = matML(pi, aln.root, leaves, edges, tm_host, *args)
        del cache
    barrier()
    eng.sync()
    s0 = eng.stats()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        l2, cache = matML(pi, aln.root, leaves, edges, tm_host, *args)
        del cache
    e2e_s = (time.perf_counter() - t0) / a.steps
    s1 = eng.stats()
    e2e_s = _max_over_ranks(dist, e2e_s)
    assert abs(l2 - lnl) <= 1e-12 * abs(lnl), (l2, lnl)
    e2e = {"value": 1.0 / e2e_s, "unit": UNIT, "h2d_bytes_per_step": (s1["h2d_bytes"] - s0["h2d_bytes"]) / a.steps,
           "d2h_bytes_per_step": (s1["d2h_bytes"] - s0["d2h_bytes"]) / a.steps,
           "note": "tips are resident (uploaded once by the first call, like the reference's LEAF_LLMAT); per step: "
                   "host P matrices + op list in, lnL out"}

    # The same call fed the way this package's own drop-in modules feed it: get_prob_t_all builds the tables on the
    # device from (pi, rates, branch lengths), matML takes the device tables -- what the unchanged reference driver
    # does on the compat modules.  Reported next to `e2e` (which keeps reference-style HOST matrices as its input).
    from cybayes_b200.subst import get_prob_t_all
    for _ in range(3):
        tabs = get_prob_t_all(pi, aln.tree, aln.er, aln.rates)
        l3, cache = matML(pi, aln.root, leaves, edges, tabs, *args)
        del cache, tabs
    barrier()
    eng.sync()
    s0 = eng.stats()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        tabs = get_prob_t_all(pi, aln.tree, aln.er, aln.rates)
        l3, cache = matML(pi, aln.root, leaves, edges, tabs, *args)
        del cache, tabs
    dev_s = (time.perf_counter() - t0) / a.steps
    s1 = eng.stats()
    dev_s = _max_over_ranks(dist, dev_s)
    assert abs(l3 - lnl) <= 1e-9 * abs(lnl), (l3, lnl)
    e2e["device_built_tables"] = {"value": 1.0 / dev_s, "unit": UNIT,
                                  "h2d_bytes_per_step": (s1["h2d_bytes"] - s0["h2d_bytes"]) / a.steps,
                                  "d2h_bytes_per_step": (s1["d2h_bytes"] - s0["d2h_bytes"]) / a.steps,
                                  "note": "get_prob_t_all (P(t) built on the device, one launch) + matML per step"}

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config_dict(a),
        "lnL": lnl, "wall_ms_per_step": wall_ms / a.steps, "host_ms_per_step": ms_per_step - statistics.mean(kernel_ms),
        "host_us_per_eval_rank0": host_prof,
        "roofline": roofline, "e2e": e2e,
        "gpu_launches": st1["kernel_launches"] - st0["kernel_launches"], "clocks": clock_rec,
        "data_generation_s": t_gen,
    }

    if not a.no_extras:
        # MCMC generations/s on THIS alignment (all ranks: every evaluation of a sharded chain is collective): the
        # generation loop inside the library (cb_chain_*), GTR + Gamma-4 moves of mat_mcmc_gamma.py:65-84
        try:
            out["mcmc_on_workload"] = mcmc_on_workload(eng, aln, pi, dist, n_gen=max(40, min(400, 20 * a.steps)))
        except Exception as exc:  # extras must never sink the headline number
            out["mcmc_on_workload"] = {"error": repr(exc)}

    if rank == 0 and world == 1 and not a.no_extras:
        # dirty-path evaluations (cache_matML's job) on the same alignment: random tip -> root paths
        l_full, snap = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True)
        parents = {c: p for (p, c) in aln.tree}
        rng = np.random.default_rng(5)
        paths = []
        for tip in rng.integers(1, N + 1, size=24):
            path, n = [], int(tip)
            while n != aln.root:
                n = parents[n]
                path.append(n)
            path.sort(key=plan.index.__getitem__)
            nodes = np.array(path, dtype=np.int32)
            ch = np.array([c for n in path for c in plan.kids[n]], dtype=np.int32)
            ps = np.array([[slot_of[k, (n, c)] for k in range(C)] for n in path for c in plan.kids[n]], dtype=np.int32)
            paths.append((nodes, ch, ps))
        ms, req = [], []
        for nodes, ch, ps in paths:
            l_d, s2 = eng.eval(snap, nodes, ch, ps, pi, want_snapshot=True)
            ms.append(eng.last_eval_main_ms())
            i2 = eng.last_eval_info()
            req.append(i2["bytes_written"] + i2["bytes_read"])
            eng.release_snapshot(s2)
            assert l_d == l_full
        mean_len = statistics.mean(len(p[0]) for p in paths)
        d_ms, d_req = statistics.mean(ms[2:]), statistics.mean(req[2:])
        out["dirty_path"] = {"evals_per_sec": 1e3 / d_ms, "mean_path_nodes": mean_len, "kernel_ms": d_ms,
                             "launches_per_eval": 2 if n_local >= 75776 else 1,
                             "roofline": {"bound": "hbm", "required_bytes_per_eval": d_req,
                                          "achieved": d_req / (d_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                          "frac": d_req / (d_ms * 1e-3) / 1e9 / peak},
                             "check": "each equals the full-pass lnL bit for bit"}
        eng.release_snapshot(snap)
        # likelihood only (no cache kept): what a proposal that is going to be rejected costs
        ms = []
        for _ in range(6):
            l_only, _ = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=False)
            ms.append(eng.last_eval_main_ms())
        assert l_only == l_full
        i3 = eng.last_eval_info()
        out["lnl_only"] = {"evals_per_sec": 1e3 / statistics.mean(ms[2:]), "kernel_ms": statistics.mean(ms[2:]),
                           "required_bytes_per_eval": i3["bytes_written"] + i3["bytes_read"],
                           "note": "same walk, nothing stored except the partials the walk itself re-reads"}

    if rank == 0 and world == 1 and not a.no_extras:
        # CPU baseline beside it: the compiled reference, 1 core, on one 125 000-site chunk of the same data -- and the
        # parity check of BASELINE.md plan step 4: that chunk through the SAME kernel instantiation (>= 75 776
        # patterns) with the reference's own P matrices, single-launch walk and split walk.
        chunk = min(BLOCK, n_local)
        base, ref_lnl, ref_mats = cpu_baseline_chunk(a, S, SEED, BLOCK, chunk)
        out["cpu_baseline"] = base
        if ref_lnl is not None:
            from cybayes_b200.engine import Engine
            e2 = Engine(np.ascontiguousarray(codes[:, :chunk]), S, C, device=local)
            b2 = e2.alloc_slots(n_e * C)
            e2.upload_pmats(np.arange(b2.base, b2.base + n_e * C, dtype=np.int32), ref_mats)
            ps2 = pslots - block.base + b2.base
            got_walk, _ = e2.eval(None, plan.nodes, plan.children, ps2, pi, want_snapshot=False, force_walk=True)
            got_split, sn = e2.eval(None, plan.nodes, plan.children, ps2, pi, want_snapshot=True)
            launches = e2.last_eval_info()["launches"]
            e2.close()
            out["cpu_baseline"]["parity"] = {
                "chunk_sites": chunk, "chunk_lnL_reference": ref_lnl, "chunk_lnL_gpu_single_walk": got_walk,
                "chunk_lnL_gpu_default_schedule": got_split, "default_schedule_launches": launches,
                "rel_err": abs(got_walk - ref_lnl) / abs(ref_lnl),
                "rel_err_default_schedule": abs(got_split - ref_lnl) / abs(ref_lnl),
                "note": "same kernel instantiation as the timed run; P matrices are the reference's own (scipy expm)"}
        # MCMC generations/s through the driver on the reference's README example (config C1)
        try:
            import io
            from cybayes_b200.driver import run_chain
            likelihood.reset_engines()
            os.environ["CYBAYES_COMPRESS_MAX_SITES"] = "250000"
            likelihood.COMPRESS_MAX_SITES = 250000
            from cybayes_b200.fastchain import run_chain_native
            res = run_chain(os.path.join(DATA, "narrow.phy"), "F81", 3000, 1000, "bin",
                            os.path.join(tempfile.gettempdir(), "bench_narrow"), out=io.StringIO())
            likelihood.reset_engines()
            nat = run_chain_native(os.path.join(DATA, "narrow.phy"), "F81", 10000, 1000, "bin",
                                   os.path.join(tempfile.gettempdir(), "bench_narrow_native"), out=io.StringIO())
            out["mcmc"] = {"gens_per_sec": nat["gens_per_sec"], "driver_py_gens_per_sec": res["gens_per_sec"],
                           "config": "C1 narrow.phy F81 bin Gamma-4: 10 000 generations with the loop inside the library "
                                     "(cb_chain_run), 3 000 through cybayes_b200.driver (Python loop); both take the "
                                     "reference driver's decisions generation by generation (tests)",
                           "final_lnL": float(nat["state"]["logLikehood"]),
                           "driver_py_final_lnL": float(res["state"]["logLikehood"])}
        except Exception as exc:  # extras must never sink the headline number
            out["mcmc"] = {"error": repr(exc)}
    elif rank == 0:
        out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 1, "kind": "reference",
                               "sample": "reported at N=1 only"}

    if rank == 0:
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------- C5
def mcmc_on_workload(eng, aln, pi, dist, n_gen, seed=1234):
    """n_gen Metropolis-Hastings generations on the bench alignment with the generation loop inside the library
    (fastchain.NativeChain over the engine's own context).  Sharded runs: every rank runs the same chain (same seeds,
    and the cross-GPU sum gives every rank the same bits), so the decisions agree without any further exchange.
    The binary GTR model has a single exchangeability: its `rates` block is left out (SURVEY F5, the reference would
    crash proposing it)."""
    import random
    from cybayes_b200 import config
    from cybayes_b200.fastchain import MOVES, NativeChain
    from cybayes_b200.ML_gamma import matML
    from cybayes_b200.subst import get_prob_t_all
    random.seed(seed)
    np.random.seed(seed)
    state = {"tree": dict(aln.tree), "pi": np.array(pi, dtype=np.float64), "rates": np.array(aln.er, dtype=np.float64),
             "srates": float(aln.alpha), "root": aln.root}
    chain = NativeChain(eng, state, list(aln.rates), "GTR", True, skip_degenerate_rates=True)
    chain.take_rng()
    chain.run(min(20, n_gen))                     # warm-up: plan cache, buffer pool
    if dist is not None:
        dist.barrier()
    eng.sync()
    t0 = time.perf_counter()
    mv, acc, cur, prop, ratio, logu = chain.run(n_gen)
    secs = _max_over_ranks(dist, time.perf_counter() - t0)
    st = chain.state()
    counts = {MOVES[m][1] + ":" + MOVES[m][0]: [int((mv == m).sum()), int(acc[mv == m].sum())] for m in np.unique(mv)}
    chain.give_rng()
    chain.close()
    # the chain's likelihood of its final state against a fresh full evaluation of that state
    tabs = get_prob_t_all(st["pi"], st["tree"], st["rates"], st["site_rates"])
    from cybayes_b200.tree import adjlist2nodes_dict, postorder
    edges = postorder(adjlist2nodes_dict(st["tree"]), aln.root)[::-1]
    fresh, cache = matML(st["pi"], aln.root, config.LEAF_LLMAT, edges, tabs, config.N_SITES, config.N_TAXA, len(tabs))
    del cache, tabs
    rel = abs(float(fresh) - float(st["logLikehood"])) / abs(float(fresh))
    assert rel <= 1e-9, (fresh, st["logLikehood"])
    return {"gens_per_sec": n_gen / secs, "generations": n_gen, "ms_per_generation": 1e3 * secs / n_gen,
            "moves_proposed_accepted": counts, "final_lnL": float(st["logLikehood"]),
            "final_lnL_vs_fresh_full_evaluation_rel": rel,
            "note": "cb_chain_run on the bench alignment (GTR + Gamma-4 move mix of mat_mcmc_gamma.py:65-84 without the "
                    "degenerate rates block); branch / NNI / SPR proposals are dirty-path evaluations, pi / alpha "
                    "proposals full passes"}


def run_c5(a):
    """C5: 512 taxa x 200 000 patterns x 64 states, GTR + Gamma-4 (FP64 tensor path, prune_dmma_rc_kernel<64>).
    On one GPU the full cache (209 GB) does not fit: the step is the likelihood-only evaluation there; sharded
    over N >= 2 GPUs (torchrun) the step keeps the cache."""
    rank, world, local, dist = _rendezvous(a)
    from cybayes_b200 import config, likelihood
    from cybayes_b200.alignment import LeafMatrices
    from cybayes_b200.ML_gamma import matML
    from cybayes_b200.synthetic import SyntheticAlignment, shard_bounds
    S, C, N = 64, 4, a.taxa
    block_sites = min(a.patterns, 25000)
    aln = SyntheticAlignment(N, a.patterns, S, 20260102, block_sites=block_sites)
    lo, hi = shard_bounds(a.patterns, rank, world, block_sites)
    t_gen = time.perf_counter()
    codes = aln.codes(lo, hi)
    t_gen = time.perf_counter() - t_gen
    n_local = hi - lo
    config.N_TAXA, config.N_CHARS, config.N_SITES, config.MODEL, config.IN_DTYPE = N, S, n_local, "GTR", "multi"
    leaves = LeafMatrices(codes, S, np.ones((1, S)))
    config.LEAF_LLMAT = leaves
    eng, _ = likelihood.engine_for(leaves, C)
    if world > 1:
        box = [eng.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        eng.comm_init(box[0], rank, world)
    edges = aln.edge_order()
    plan = likelihood._plan_for(edges)
    block, slots, pslots, slot_of, ekeys = _tables(eng, aln, plan, C)
    n_e = len(ekeys)
    pi = aln.pi
    keep_cache = (N - 2) * C * S * n_local * 8 <= 150e9

    kept = []

    def step(keep=False):
        lnl, snap = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=keep_cache)
        if keep:
            kept.append(snap)
        elif snap >= 0:
            eng.release_snapshot(snap)
        return lnl

    def barrier():
        if dist is not None:
            dist.barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    for _ in range(a.warmup):
        lnl = step()
    barrier()
    eng.sync()
    if clocks:
        clocks.begin()
    st0 = eng.stats()
    kernel_ms, main_ms = [], []
    eng.mark(0)
    for i in range(a.steps):
        lnl = step(keep=a.dump_outputs is not None and i == a.steps - 1)
        kernel_ms.append(eng.last_eval_ms())
        main_ms.append(eng.last_eval_main_ms())
    eng.mark(1)
    eng.sync()
    dev_ms = eng.mark_elapsed_ms()
    st1 = eng.stats()
    info = eng.last_eval_info()
    barrier()
    clock_rec = clocks.stop() if clocks else None
    if kept:
        if rank == 0:
            dump_outputs(a.dump_outputs, eng, kept[0], lnl, plan.nodes[:-1])
        if kept[0] >= 0:
            eng.release_snapshot(kept[0])
    dev_ms = _max_over_ranks(dist, dev_ms)
    ms_per_step = dev_ms / a.steps
    n_int_edges = sum(1 for (p, c) in ekeys if c > N)
    flops = C * n_local * (2.0 * S * S * n_int_edges + S * (N - 1) + 2.0 * S)     # SURVEY 8(d), this rank's shard
    k_ms = statistics.mean(main_ms)
    fp64_peak, fp64_src = eng.fp64_peak_tflops(), "measured in this run (cb_fp64_peak: DMMA m8n8k4 from registers)"
    hbm_peak, hbm_src = measured_peaks()
    required = info["bytes_written"] + info["bytes_read"]
    roofline = {"bound": "tensor", "achieved": flops / (k_ms * 1e-3) / 1e12, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": flops / (k_ms * 1e-3) / 1e12 / fp64_peak, "traffic": None, "kernel": "prune_dmma_rc_kernel<64, true>",
                "algorithmic_flop_per_eval": flops, "kernel_ms_per_eval": k_ms, "peak_source": fp64_src,
                "note": "FP64 tensor (mma.sync DMMA; tcgen05 has no fp64 kind)",
                "hbm": {"required_bytes_per_eval": required, "GBps": required / (k_ms * 1e-3) / 1e9, "peak": hbm_peak,
                        "frac": required / (k_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src},
                "op_list": {k: info[k] for k in ("ops", "stored", "read_back", "launches")}}
    # end to end: reference-style host P dicts -> matML
    host_p = eng.download_pmats(slots).reshape(C, n_e, S, S)
    tm_host = [{e: host_p[k, i] for i, e in enumerate(ekeys)} for k in range(C)]
    for _ in range(2):
        l2, cache = matML(pi, aln.root, leaves, edges, tm_host, n_local, N, C)
        del cache
    barrier()
    eng.sync()
    s0 = eng.stats()
    t0 = time.perf_counter()
    n_e2e = max(3, a.steps // 4)
    for _ in range(n_e2e):
        l2, cache = matML(pi, aln.root, leaves, edges, tm_host, n_local, N, C)
        del cache
    e2e_s = _max_over_ranks(dist, (time.perf_counter() - t0) / n_e2e)
    s1 = eng.stats()
    assert abs(l2 - lnl) <= 1e-12 * abs(lnl), (l2, lnl)
    out = {"metric": METRIC, "value": 1e3 / ms_per_step, "unit": UNIT, "n_gpus": world, "steps": a.steps,
           "warmup": a.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(a), "lnL": lnl,
           "cache_kept": bool(keep_cache), "roofline": roofline,
           "e2e": {"value": 1.0 / e2e_s, "unit": UNIT, "h2d_bytes_per_step": (s1["h2d_bytes"] - s0["h2d_bytes"]) / n_e2e,
                   "d2h_bytes_per_step": (s1["d2h_bytes"] - s0["d2h_bytes"]) / n_e2e,
                   "note": "host P matrices (134 MB) + op list in, lnL out; matML keeps the cache when it fits, else "
                           "evaluates the likelihood and materialises the cache on first use"},
           "gpu_launches": st1["kernel_launches"] - st0["kernel_launches"], "clocks": clock_rec,
           "data_generation_s": t_gen}
    if rank == 0 and world == 1 and not a.no_extras:
        chunk = min(2000, n_local)
        base, ref_lnl, ref_mats = cpu_baseline_chunk(a, S, 20260102, block_sites, chunk, reps=2)
        out["cpu_baseline"] = base
        if ref_lnl is not None:
            from cybayes_b200.engine import Engine
            os.environ["CYBAYES_DMMA_RC"] = "1"
            e2 = Engine(np.ascontiguousarray(aln.codes(0, block_sites)[:, :chunk]), S, C, device=local)
            del os.environ["CYBAYES_DMMA_RC"]
            b2 = e2.alloc_slots(n_e * C)
            e2.upload_pmats(np.arange(b2.base, b2.base + n_e * C, dtype=np.int32), ref_mats)
            got, _ = e2.eval(None, plan.nodes, plan.children, pslots - block.base + b2.base, pi, want_snapshot=False)
            e2.close()
            out["cpu_baseline"]["parity"] = {"chunk_sites": chunk, "chunk_lnL_reference": ref_lnl, "chunk_lnL_gpu": got,
                                             "rel_err": abs(got - ref_lnl) / abs(ref_lnl)}
    elif rank == 0:
        out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 1, "kind": "reference", "sample": "reported at N=1 only"}
    if rank == 0:
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------ C1 - C3
def _reference_real(fname, reader, dtype, model, n_gen):
    """The compiled reference, 1 core, fresh interpreter: ms per full matML / cache_matML and generations/s of its
    own driver loop on the real dataset."""
    code = f'''
import sys, io, time, random, contextlib, json, runpy
import numpy as np
sys.path.insert(0, {os.path.join(REPO, "oracle", "_ref")!r})
import config, utils, mcmc_gamma, ML_gamma
np.random.seed(1234); random.seed(1234)
with contextlib.redirect_stdout(io.StringIO()):
    (config.N_TAXA, config.N_CHARS, config.ALPHABET, sd, config.LEAF_LLMAT, config.TAXA, config.N_SITES) = utils.{reader}({os.path.join(DATA, fname)!r})
config.IN_DTYPE, config.MODEL, config.N_NODES = {dtype!r}, {model!r}, 2 * config.N_TAXA - 1
st = mcmc_gamma.state_init()
a = (config.N_SITES, config.N_TAXA, config.N_CATS)
lnl, cache = ML_gamma.matML(st["pi"], st["root"], config.LEAF_LLMAT, st["postorder"], st["transitionMat"], *a)
t = []
for _ in range(5):
    t0 = time.perf_counter(); ML_gamma.matML(st["pi"], st["root"], config.LEAF_LLMAT, st["postorder"], st["transitionMat"], *a); t.append(time.perf_counter() - t0)
rev = mcmc_gamma.adjlist2reverse_nodes_dict(st["tree"])
td = []
rng = random.Random(3)
for _ in range(20):
    p, c = rng.choice(list(st["tree"]))
    path = mcmc_gamma.get_path2root(rev, c, st["root"])
    t0 = time.perf_counter(); ML_gamma.cache_matML(st["pi"], st["root"], config.LEAF_LLMAT, cache, path, st["postorder"], st["transitionMat"], *a); td.append(time.perf_counter() - t0)
gps = None
if {reader!r} != "readPhy":
    sys.argv = ["mat_mcmc_gamma.py", "-i", {os.path.join(DATA, fname)!r}, "-m", {model!r}, "-n", "{n_gen}", "-t", "1000", "-d", {dtype!r}, "-o", "/tmp/bench_ref_real"]
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        runpy.run_path({os.path.join(REPO, "oracle", "_ref", "mat_mcmc_gamma.code")!r}, run_name="__main__")
    gps = {n_gen} / (time.perf_counter() - t0)
print("@@" + json.dumps([sorted(t)[len(t)//2] * 1e3, sum(td) / len(td) * 1e3, float(lnl), gps]))
'''
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    line = [l for l in res.stdout.splitlines() if l.startswith("@@")]
    return json.loads(line[0][2:]) if line else None


def run_real(a):
    """C1 - C3: the real datasets (latency-bound, cache 8-90 MB).  metric = MCMC generations/s through the restated
    driver on the CUDA engine (value, fast driver; e2e = the reference's own unmodified script on the compat
    modules where its reader can parse the file), with us per full / dirty-path evaluation and batched proposal
    scoring beside it."""
    import io
    import random
    from cybayes_b200 import config, likelihood
    from cybayes_b200.driver import load_alignment, run_chain
    from cybayes_b200.mcmc_gamma import adjlist2reverse_nodes_dict, get_path2root, state_init
    from cybayes_b200.ML_gamma import cache_matML, matML
    os.environ["CYBAYES_COMPRESS_MAX_SITES"] = "250000"
    likelihood.COMPRESS_MAX_SITES = 250000
    fname, reader, dtype, model = REAL[a.config]
    likelihood.reset_engines()
    np.random.seed(1234)
    random.seed(1234)
    load_alignment(os.path.join(DATA, fname), dtype, reader)
    config.MODEL = model
    st = state_init()
    args = (config.N_SITES, config.N_TAXA, config.N_CATS)
    lnl, cache = matML(st["pi"], st["root"], config.LEAF_LLMAT, st["postorder"], st["transitionMat"], *args)
    eng, _ = likelihood.engine_for(config.LEAF_LLMAT, config.N_CATS)
    clocks = ClockSampler(int(os.environ.get("CYBAYES_DEVICE", "0")))
    wall, dev = [], []
    for _ in range(a.warmup + 30):
        t0 = time.perf_counter()
        l2, c2 = matML(st["pi"], st["root"], config.LEAF_LLMAT, st["postorder"], st["transitionMat"], *args)
        wall.append(time.perf_counter() - t0)
        dev.append(eng.last_eval_ms())
        del c2
    info_full = eng.last_eval_info()
    parents = adjlist2reverse_nodes_dict(st["tree"])
    rng = random.Random(3)
    dwall, ddev, dlen = [], [], []
    for _ in range(40):
        p, c = rng.choice(list(st["tree"]))
        path = get_path2root(parents, c, st["root"])
        t0 = time.perf_counter()
        l3, c3 = cache_matML(st["pi"], st["root"], config.LEAF_LLMAT, cache, path, st["postorder"], st["transitionMat"], *args)
        dwall.append(time.perf_counter() - t0)
        ddev.append(eng.last_eval_ms())
        dlen.append(len(path))
        assert l3 == lnl
        del c3
    wall, dev = wall[a.warmup:], dev[a.warmup:]
    n_states, n_patterns, n_taxa, n_sites = config.N_CHARS, eng.n_patterns, config.N_TAXA, config.N_SITES
    likelihood.reset_engines()
    n_gen = a.steps if a.steps is not None else {"C1": 20000, "C2": 4000, "C3": 4000}[a.config]
    res = run_chain(os.path.join(DATA, fname), model, n_gen, 1000, dtype, os.path.join(tempfile.gettempdir(), "b_" + a.config),
                    reader=reader, out=io.StringIO(), fast_spr=True)
    gens = res["gens_per_sec"]
    fast, timed = None, res
    try:
        from cybayes_b200.fastchain import run_chain_native
        likelihood.reset_engines()
        r2 = run_chain_native(os.path.join(DATA, fname), model, n_gen, 1000, dtype,
                              os.path.join(tempfile.gettempdir(), "bn_" + a.config), reader=reader, out=io.StringIO())
        fast = {"gens_per_sec": r2["gens_per_sec"], "same_final_lnL": float(r2["state"]["logLikehood"]) == float(res["state"]["logLikehood"])}
        timed = r2
    except ImportError:
        pass
    if a.dump_outputs is not None:
        dump_chain_state(a.dump_outputs, timed["state"])
    clock_rec = clocks.stop()
    peak, peak_src = measured_peaks()
    req = info_full["bytes_written"] + info_full["bytes_read"]
    d_us = statistics.median(dev) * 1e3
    ref = _reference_real(fname, reader, dtype, model, min(n_gen, 3000)) if reference_available() and not a.no_extras else None
    value = fast["gens_per_sec"] if fast else gens
    out = {"metric": "MCMC generations/sec", "value": value, "unit": "gens/s", "n_gpus": 1, "steps": n_gen, "warmup": a.warmup,
           "ms_per_step": 1e3 / value, "higher_is_better": True, "scaling": "replicas only", "vs_baseline": None,
           "dtype": "f64", "data": f"tests/golden/data/{fname} (reference dataset)",
           "config": {"workload": f"{a.config}: {fname} {model} + Gamma-4 MCMC, {n_gen} generations, seed 1234",
                      "n_taxa": n_taxa, "n_sites": n_sites, "n_patterns": n_patterns, "n_states": n_states,
                      "l2": "whole partial cache is L2-resident (8-90 MB): latency-bound, no flush"},
           "driver_py": {"gens_per_sec": gens, "note": "cybayes_b200.driver (restated MH loop, Python) with dirty-path SPR"},
           "native_loop": fast,
           "full_eval": {"device_us": d_us, "call_us": statistics.median(wall) * 1e6},
           "dirty_path": {"device_us": statistics.median(ddev) * 1e3, "call_us": statistics.median(dwall) * 1e6,
                          "mean_path_nodes": statistics.mean(dlen)},
           "roofline": {"bound": "hbm", "achieved": req / (d_us * 1e-6) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": req / (d_us * 1e-6) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                        "note": "launch-latency-bound (SURVEY 8d): the cache is L2-resident; absolute us per "
                                "evaluation is the figure of merit, the fraction is given for completeness"},
           "e2e": {"value": value, "unit": "gens/s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": 8,
                   "note": "every generation uploads op descriptors + new P scalars and reads lnL back"},
           "clocks": clock_rec, "lnL_initial": float(lnl)}
    if ref:
        out["cpu_baseline"] = {"value": ref[3], "unit": "gens/s", "cores": 1, "kind": "reference",
                               "sample": f"the reference's own driver, {min(n_gen, 3000)} generations, 1 core "
                                         "(None where its reader cannot parse the file, SURVEY F4)",
                               "full_eval_ms": ref[0], "dirty_path_ms": ref[1],
                               "lnL_rel_err": abs(float(lnl) - ref[2]) / abs(ref[2])}
    print(json.dumps(out))


def main():
    a = parse()
    if a.impl == "reference":
        if a.config in REAL:
            print(json.dumps({"impl": "reference", "unavailable": "the reference arm of C1-C3 is reported inside "
                              "cpu_baseline of the --config line (its driver is single-process)"}))
            return
        run_reference_arm(a)
    elif a.config == "C4":
        run_c4(a)
    elif a.config == "C5":
        run_c5(a)
    else:
        run_real(a)


if __name__ == "__main__":
    main()
