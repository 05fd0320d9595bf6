"""Posterior predictive replicates (simulate_kernel, cb_simulate, Engine.simulate, ppc.Replicates, the drivers' --ppc).

CPU: a NumPy restatement of the simulator -- Philox4x32-10 checked against the Random123 known answers -- whose column
pattern frequencies match the exact pattern probabilities of the pruning oracle (chi-square); the mask, edge-order and
column-offset properties; both drivers writing .ppc on an oracle-backed fake engine whose cb_simulate is the
restatement, with .log, .trees and stdout unchanged; the refusal under sharding; and the kernel ledger of the whole
binary (test_kernel_coverage.py keeps the ledger of the top-level csrc/ sources, this file the one of csrc/ppc/).
GPU: every ledger kernel under the profiler, cb_simulate against the restatement byte for byte, the replicate's lnL and
T against a fresh context, the P / tree mapping of the replicate context, the snapshot refusal and the drivers."""
import io
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
from scipy.stats import chi2

import pruning_oracle as oracle
from conftest import REPO
from fake_engine import FakeEngine

NARROW = os.path.join(REPO, "tests", "golden", "data", "narrow.phy")
CSRC = os.path.join(REPO, "cybayes_b200", "csrc")
U8, U16 = np.uint8, np.uint16

# kernels of csrc/ppc/: name -> code dtype of the case that launches it
PPC_LEDGER = {"simulate_kernel<unsigned char>": U8, "simulate_kernel<unsigned short>": U16}

# ------------------------------------------------------------------------------------------- NumPy restatement
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 on uint32 values held in uint64 arrays: ctr = 4 arrays (broadcastable), key = 2 ints."""
    c0, c1, c2, c3 = (np.asarray(x, dtype=np.uint64) for x in ctr)
    k0, k1 = np.uint64(key[0]), np.uint64(key[1])
    m0, m1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2          # < 2^64: exact
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _MASK
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _MASK, (k1 + np.uint64(0xBB67AE85)) & _MASK
    return c0, c1, c2, c3


def _pick(rows, x):
    """Inverse CDF: the first j with u < row[0] + ... + row[j] (fp64, left to right), else S - 1."""
    S = rows.shape[-1]
    u = (x.astype(np.float64) + 0.5) * 2.0 ** -32
    hit = u[:, None] < np.cumsum(rows[:, :S - 1], axis=1)
    return np.where(hit.any(axis=1), hit.argmax(axis=1), S - 1)


def simulate_restated(codes, S, C, parents, children, pslots, pool, pi, root, seed, replicate, column_offset=0,
                      chunk=8192):
    """The replicate cb_simulate writes, restated: codes (n_taxa, n_sites) -> new array; pool: slot -> (S, S)."""
    codes = np.array(codes, copy=True)
    n_taxa, n_sites = codes.shape
    key = (seed & 0xFFFFFFFF, seed >> 32)
    mats = [np.stack([pool[int(s)] for s in row]) for row in np.asarray(pslots)]   # per edge: (C, S, S)
    n_blocks = (2 + 2 * n_taxa) // 4 + 1
    for lo in range(0, n_sites, chunk):
        hi = min(n_sites, lo + chunk)
        col = np.arange(lo, hi, dtype=np.uint64) + np.uint64(column_offset)
        words = np.stack(philox4x32_10((np.arange(n_blocks, dtype=np.uint64)[:, None], (col & _MASK)[None],
                                        (col >> np.uint64(32))[None], np.uint64(replicate)), key), axis=1)

        def draw(k):
            return words[k // 4, k % 4]
        cat = ((draw(0) * np.uint64(C)) >> np.uint64(32)).astype(np.int64)
        state = {int(root): _pick(np.broadcast_to(np.asarray(pi, dtype=np.float64), (hi - lo, S)), draw(1))}
        for e, (p, ch) in enumerate(zip(np.asarray(parents).tolist(), np.asarray(children).tolist())):
            s = _pick(mats[e][cat, state[p]], draw(1 + ch))
            if ch <= n_taxa:
                row = codes[ch - 1, lo:hi]
                m = row < S
                row[m] = s[m]
            else:
                state[ch] = s
    return codes


def _preorder(tree, root):
    out, stack = [], [root]
    kids = oracle.children_of(tree)
    while stack:
        n = stack.pop()
        for c in kids.get(n, ()):
            out.append((n, c))
            stack.append(c)
    return out


# ------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    """The Random123 known-answer vectors of Philox4x32-10."""
    assert tuple(int(x) for x in philox4x32_10(ctr, key)) == want


def _small_problem(S, C, n_taxa, seed):
    rng = np.random.default_rng(seed)
    tree, nodes, nxt = {}, list(range(1, n_taxa + 1)), n_taxa + 1
    while len(nodes) > 1:
        a, b = nodes.pop(int(rng.integers(len(nodes)))), nodes.pop(int(rng.integers(len(nodes))))
        tree[nxt, a], tree[nxt, b] = float(rng.exponential(0.3)), float(rng.exponential(0.3))
        nodes.append(nxt)
        nxt += 1
    root = nxt - 1
    pi = rng.dirichlet(np.full(S, 3.0))
    er = rng.dirichlet(np.ones(S * (S - 1) // 2))
    rates = oracle.site_rates(0.5, C) if C > 1 else [1.0]
    tm = [oracle.prob_t("GTR", False, pi, tree, er, r) for r in rates]
    pre = _preorder(tree, root)
    pool, pslots = {}, []
    for i, e in enumerate(pre):
        pslots.append([i * C + k for k in range(C)])
        for k in range(C):
            pool[i * C + k] = tm[k][e]
    return tree, root, pi, tm, pre, pool, np.array(pslots, dtype=np.int32)


@pytest.mark.parametrize("S,n_taxa", [(2, 5), (4, 4)])
@pytest.mark.parametrize("C", [1, 4])
def test_sampler_samples_the_model(S, n_taxa, C):
    """2^20 simulated columns: their pattern counts against the exact pattern probabilities of the pruning oracle over
    all S^N patterns (chi-square, cells with an expectation below 5 pooled; fixed seed, fixed threshold)."""
    tree, root, pi, tm, pre, pool, pslots = _small_problem(S, C, n_taxa, 100 * S + C)
    n = 1 << 20
    sim = simulate_restated(np.zeros((n_taxa, n), dtype=U8), S, C, [p for p, _ in pre], [c for _, c in pre], pslots,
                            pool, pi, root, seed=0x1234_5678_9abc_def0, replicate=7, chunk=1 << 16)
    weights = S ** np.arange(n_taxa - 1, -1, -1)
    counts = np.bincount(weights @ sim.astype(np.int64), minlength=S ** n_taxa)
    patterns = np.array(np.unravel_index(np.arange(S ** n_taxa), (S,) * n_taxa), dtype=np.int64)
    leaves = {t + 1: np.eye(S)[patterns[t]].T for t in range(n_taxa)}
    edges = oracle.edge_order(tree, root, n_taxa)
    _, per_site = oracle.mat_ml_scaled(pi, root, leaves, edges, tm, S ** n_taxa, n_taxa, n_cats=C, site_lnl=True)
    prob = np.exp(per_site)
    assert abs(prob.sum() - 1.0) < 1e-12
    expected = prob * n
    big = expected >= 5
    obs = np.append(counts[big], counts[~big].sum())
    exp = np.append(expected[big], expected[~big].sum())
    if exp[-1] == 0:
        obs, exp = obs[:-1], exp[:-1]
    stat = float(np.sum((obs - exp) ** 2 / exp))
    p = chi2.sf(stat, len(obs) - 1)
    assert p > 1e-4, (stat, len(obs) - 1, p)


def _masked_problem(S=4, C=2, n_taxa=9, n_sites=300, dtype=U8, seed=3):
    from test_gpu_parity import _random_problem
    tree, root, _, codes, amb, pi, er, rates = _random_problem(seed, n_taxa, n_sites, S, n_cats=C, code_dtype=dtype)
    tm = [oracle.prob_t("GTR", False, pi, tree, er, r) for r in rates]
    pre = _preorder(tree, root)
    pool = {i * C + k: tm[k][e] for i, e in enumerate(pre) for k in range(C)}
    pslots = np.array([[i * C + k for k in range(C)] for i in range(len(pre))], dtype=np.int32)
    return dict(tree=tree, root=root, codes=codes, amb=amb, pi=pi, tm=tm, pre=pre, pool=pool, pslots=pslots, S=S, C=C)


def _check_properties(simulate, p, seed=99, replicate=3):
    """simulate(codes, parents, children, pslots, replicate, column_offset) -> replicate codes.  The mask is kept and
    simulating again into a replicate changes nothing; the edge order does not matter; column-offset slices concatenate
    to the whole; another replicate id gives another replicate."""
    codes, S, pre, ps = p["codes"], p["S"], p["pre"], p["pslots"]
    par, ch = np.array([a for a, _ in pre]), np.array([b for _, b in pre])
    whole = simulate(codes, par, ch, ps, replicate, 0)
    assert whole.dtype == codes.dtype and whole.shape == codes.shape
    assert np.array_equal(whole >= S, codes >= S) and np.array_equal(whole[codes >= S], codes[codes >= S])
    assert (whole < S).any() and not np.array_equal(whole, codes)
    assert np.array_equal(simulate(whole, par, ch, ps, replicate, 0), whole)
    # another parents-first order: the root's subtrees swapped, every node's children reversed (BFS)
    order = []
    frontier = [p["root"]]
    kids = oracle.children_of(p["tree"])
    while frontier:
        nxt = []
        for n in frontier:
            for c in reversed(kids.get(n, ())):
                order.append(pre.index((n, c)))
                nxt.append(c)
        frontier = nxt
    order = np.array(order)
    assert not np.array_equal(order, np.arange(len(pre)))
    assert np.array_equal(simulate(codes, par[order], ch[order], ps[order], replicate, 0), whole)
    cut = 131
    parts = [simulate(np.ascontiguousarray(codes[:, lo:hi]), par, ch, ps, replicate, lo)
             for lo, hi in ((0, cut), (cut, codes.shape[1]))]
    assert np.array_equal(np.concatenate(parts, axis=1), whole)
    assert not np.array_equal(simulate(codes, par, ch, ps, replicate + 1, 0), whole)


@pytest.mark.parametrize("dtype", [U8, U16])
def test_mask_edge_order_and_column_offset(dtype):
    p = _masked_problem(dtype=dtype)

    def restated(codes, par, ch, ps, rep, off):
        return simulate_restated(codes, p["S"], p["C"], par, ch, ps, p["pool"], p["pi"], p["root"], 99, rep, off)
    _check_properties(restated, p)


def test_multinomial_statistic():
    from cybayes_b200.ppc import multinomial_statistic
    w = np.array([3.0, 1.0, 2.0])
    assert multinomial_statistic(w) == pytest.approx(3 * np.log(3) + 2 * np.log(2) - 6 * np.log(6), rel=1e-15)
    assert multinomial_statistic(np.ones(5)) == pytest.approx(-5 * np.log(5), rel=1e-15)
    assert multinomial_statistic([7.0]) == 0.0


class PPCFakeEngine(FakeEngine):
    """FakeEngine with the cb_simulate stand-in: the NumPy restatement over its codes and P pool."""

    def __init__(self, codes, n_states, n_cats, amb_sets=None, weights=None, device=None):
        super().__init__(codes, n_states, n_cats, amb_sets, weights, device)
        self.codes = np.array(codes, copy=True)
        self.amb = np.ones((1, n_states)) if amb_sets is None else np.asarray(amb_sets, dtype=float)
        self.n_simulate = 0

    def simulate(self, parents, children, pslots, pi, root, seed, replicate, column_offset=0, download=True):
        if self.snaps:
            raise RuntimeError("cb_simulate: the context holds a live snapshot")
        self.codes = simulate_restated(self.codes, self.n_states, self.n_cats, parents, children, pslots, self.pm, pi,
                                       root, int(seed), int(replicate), column_offset)
        table = np.vstack([np.eye(self.n_states), self.amb])
        self.leaves = {t + 1: np.ascontiguousarray(table[self.codes[t].astype(np.int64)].T) for t in range(self.n_taxa)}
        self.n_simulate += 1
        return self.codes.copy() if download else None


@pytest.fixture
def ppc_backend(monkeypatch):
    from cybayes_b200 import likelihood
    likelihood.reset_engines()
    likelihood._plan_cache.clear()
    monkeypatch.setattr(likelihood, "_engine_factory", PPCFakeEngine)
    FakeEngine.instances.clear()
    yield PPCFakeEngine
    likelihood.reset_engines()


def _read_ppc(path):
    lines = open(path).read().splitlines()
    return lines[0].split("\t"), [line.split("\t") for line in lines[1:]]


def _runs_with_and_without(runner, tmp_path, n_gen, thin, n_rep, seed, **kw):
    """.log, .trees and stdout byte-identical with and without --ppc; the .ppc rows in the documented format."""
    from cybayes_b200 import likelihood
    outs = {}
    for tag, n in (("plain", 0), ("ppc", n_rep)):
        likelihood.reset_engines()
        buf = io.StringIO()
        runner(NARROW, "F81", n_gen, thin, "bin", str(tmp_path / tag), out=buf, ppc=n, ppc_seed=seed, **kw)
        outs[tag] = buf.getvalue()
    for ext in (".log", ".trees"):
        assert open(str(tmp_path / ("plain" + ext)), "rb").read() == open(str(tmp_path / ("ppc" + ext)), "rb").read()
    assert outs["plain"] == outs["ppc"]
    assert not os.path.exists(str(tmp_path / "plain.ppc"))
    head, rows = _read_ppc(str(tmp_path / "ppc.ppc"))
    assert head == ["Iter", "Replicate", "LnL_obs", "LnL_rep", "T_obs", "T_rep"]
    log = [line.split("\t") for line in open(str(tmp_path / "ppc.log")).read().splitlines()[1:]]
    assert len(log) == n_gen // thin and len(rows) == len(log) * n_rep
    t_obs = {r[4] for r in rows}
    assert len(t_obs) == 1
    for i, r in enumerate(rows):
        lr = log[i // n_rep]
        assert len(r) == 6 and r[0] == lr[0] and int(r[1]) == i
        assert float(r[2]) == float(lr[1])
        assert all(x == "%.17g" % float(x) for x in r[2:])
        assert float(r[5]) <= 0.0 and float(r[3]) < 0.0
    assert len({r[3] for r in rows}) > len(rows) // 2       # replicates differ
    return open(str(tmp_path / "ppc.ppc")).read()


def test_python_driver_writes_ppc_and_nothing_else_changes(ppc_backend, tmp_path):
    from cybayes_b200.driver import run_chain
    from cybayes_b200.ppc import summary
    _runs_with_and_without(run_chain, tmp_path, 200, 20, 3, 5, fast_spr=True)
    s = summary(str(tmp_path / "ppc.ppc"), burnin=40)
    assert set(s) == {"lnL", "T"} and s["lnL"]["replicates"] == 8 * 3
    assert all(0.0 <= v["p"] <= 1.0 for v in s.values())


def test_native_loop_writes_the_same_ppc_as_the_python_driver(ppc_backend, tmp_path):
    from cybayes_b200 import likelihood
    from cybayes_b200.driver import run_chain
    from cybayes_b200.fastchain import run_chain_native
    nat = _runs_with_and_without(run_chain_native, tmp_path, 200, 20, 2, 11)
    likelihood.reset_engines()
    run_chain(NARROW, "F81", 200, 20, "bin", str(tmp_path / "py"), out=io.StringIO(), ppc=2, ppc_seed=11)
    assert open(str(tmp_path / "py.ppc")).read() == nat


def test_ppc_summary_command(ppc_backend, tmp_path, capsys):
    from cybayes_b200.driver import main
    from cybayes_b200.ppc import main as ppc_main
    main(["-i", NARROW, "-m", "F81", "-n", "40", "-t", "10", "-d", "bin", "-o", str(tmp_path / "x"), "--ppc", "2"])
    capsys.readouterr()
    ppc_main([str(tmp_path / "x.ppc")])
    out = capsys.readouterr().out.splitlines()
    assert out[0].split("\t")[0] == "statistic" and [line.split("\t")[0] for line in out[1:]] == ["lnL", "T"]
    assert all(line.split("\t")[-1] == "8" for line in out[1:])


def test_ppc_is_refused_on_a_sharded_run(monkeypatch, tmp_path, capsys):
    from cybayes_b200.driver import main
    from cybayes_b200.ppc import Replicates
    monkeypatch.setenv("CYBAYES_SHARD", "1")
    with pytest.raises(SystemExit):
        main(["-i", NARROW, "-m", "F81", "-n", "10", "-t", "5", "-d", "bin", "-o", str(tmp_path / "x"), "--ppc", "2"])
    assert "CYBAYES_SHARD=1" in capsys.readouterr().err
    with pytest.raises(ValueError, match="CYBAYES_SHARD=1"):
        Replicates({}, 4)
    assert not os.path.exists(str(tmp_path / "x.log"))


# ------------------------------------------------------------------------------------------- whole-binary ledger
def _declared(paths):
    src = "".join(open(p).read() for p in paths)
    return set(re.findall(r"__global__\s+void\s+(?:__launch_bounds__\([^)]*\)\s+)?(\w+)\s*\(", src))


def test_ledger_names_every_kernel_in_the_whole_binary():
    """Every __global__ instantiation nm finds in the library is in test_kernel_coverage's ledger, its exemptions or
    PPC_LEDGER, and every entry exists; the kernels of PPC_LEDGER are declared in csrc/ppc/."""
    from cybayes_b200 import _lib
    from test_kernel_coverage import EXEMPT, LEDGER, LIB, kernel_name
    _lib.load()
    nm = shutil.which("nm")
    if nm is None:
        pytest.skip("nm unavailable")
    ppc_dir = os.path.join(CSRC, "ppc")
    ppc_files = [os.path.join(ppc_dir, f) for f in sorted(os.listdir(ppc_dir)) if f.endswith((".cu", ".cuh"))]
    top = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh"))]
    declared, in_ppc = _declared(top + ppc_files), _declared(ppc_files)
    assert {k.split("<")[0] for k in PPC_LEDGER} <= in_ppc
    out = subprocess.run([nm, "-C", "--defined-only", LIB], capture_output=True, text=True, check=True).stdout
    found = set()
    for line in out.splitlines():
        parts = line.split(None, 2)
        if len(parts) < 3 or parts[1] not in "TtWw" or "__device_stub__" in parts[2]:
            continue
        name = kernel_name(parts[2])
        if name and name.split("<")[0] in declared:
            found.add(name)
    listed = set(LEDGER) | set(EXEMPT) | set(PPC_LEDGER)
    assert not set(PPC_LEDGER) & (set(LEDGER) | set(EXEMPT))
    assert not found - listed, f"kernels without a test case: {sorted(found - listed)}"
    assert not listed - found, f"ledger entries the binary does not contain: {sorted(listed - found)}"


# ------------------------------------------------------------------------------------------------------------ GPU
def _gpu_problem(S, C, n_taxa, n_sites, dtype=None, seed=None, tree=None):
    """Engine over a random problem with missing and polymorphic cells, P matrices uploaded; the restatement's
    inputs."""
    from cybayes_b200.engine import Engine
    from test_gpu_parity import _random_problem
    t, root, _, codes, amb, pi, er, rates = _random_problem(seed if seed is not None else 7 * S + C, n_taxa, n_sites, S,
                                                            n_cats=C, code_dtype=dtype)
    if tree is not None:
        t, root = tree
    tm = [oracle.prob_t("GTR", False, pi, t, er, r) for r in rates]
    pre = _preorder(t, root)
    eng = Engine(codes, S, C, amb)
    block = eng.alloc_slots(len(pre) * C)
    slots = np.arange(block.base, block.base + block.n, dtype=np.int32)
    eng.upload_pmats(slots, np.stack([tm[k][e] for e in pre for k in range(C)]))
    pslots = slots.reshape(len(pre), C)
    pool = {int(s): tm[k][e] for (e, row) in zip(pre, pslots) for k, s in enumerate(row)}
    return dict(eng=eng, block=block, tree=t, root=root, codes=codes, amb=amb, pi=pi, pre=pre, pool=pool,
                pslots=pslots, S=S, C=C)


def _kernel_vs_restatement(p, seed, replicate, column_offset=0):
    eng, pre = p["eng"], p["pre"]
    par, ch = [a for a, _ in pre], [b for _, b in pre]
    got = eng.simulate(par, ch, p["pslots"], p["pi"], p["root"], seed, replicate, column_offset)
    want = simulate_restated(p["codes"], p["S"], p["C"], par, ch, p["pslots"], p["pool"], p["pi"], p["root"], seed,
                             replicate, column_offset)
    assert got.dtype == p["codes"].dtype
    assert np.array_equal(got, want), np.argwhere(got != want)[:5]
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PPC_LEDGER))
def test_ppc_ledger_case(name, gpu_backend):
    """Each kernel of PPC_LEDGER is what its case launches, and nothing else of the library."""
    from test_kernel_coverage import EXEMPT, LEDGER, kernel_name
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    p = _gpu_problem(5, 2, 9, 300, dtype=PPC_LEDGER[name])
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _kernel_vs_restatement(p, 1, 0)
        torch.cuda.synchronize()
    got = {kernel_name(e.name) for e in prof.events() if e.device_type == DeviceType.CUDA}
    assert got & (set(LEDGER) | set(EXEMPT) | set(PPC_LEDGER)) == {name}, got
    p["eng"].close()


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 2, 4, 8])
@pytest.mark.parametrize("S", [2, 4, 23, 47, 64])
def test_simulate_equals_the_restatement(S, C, gpu_backend):
    """Missing and polymorphic cells, 1003 columns (ragged against the 128-column blocks and the 64-pattern padding),
    1-byte codes and the same alignment in 2-byte codes."""
    for dtype in (None, U16):
        p = _gpu_problem(S, C, 13, 1003, dtype=dtype)
        _kernel_vs_restatement(p, 0xDEADBEEF_00C0FFEE + S, 2 * C)
        p["eng"].close()


@pytest.mark.gpu
@pytest.mark.parametrize("scratch", ["0", "1"])
def test_kernel_properties(scratch, gpu_backend, monkeypatch):
    """Mask, idempotence, edge order and column-offset slices on the GPU, internal states in shared memory and in
    the global scratch."""
    from cybayes_b200.engine import Engine
    monkeypatch.setenv("CYBAYES_SIM_SCRATCH", scratch)
    p = _gpu_problem(4, 2, 9, 300, seed=3)
    p["eng"].close()

    def on_gpu(codes, par, ch, ps, rep, off):
        eng = Engine(codes, p["S"], p["C"], p["amb"])
        slots = np.unique(ps)
        eng.alloc_slots(int(slots.max()) + 1)
        eng.upload_pmats(slots, np.stack([p["pool"][int(s)] for s in slots]))
        out = eng.simulate(par, ch, ps, p["pi"], p["root"], 99, rep, off)
        eng.close()
        return out
    _check_properties(on_gpu, p)


@pytest.mark.gpu
def test_caterpillar_of_1024_taxa(gpu_backend):
    """A 1024-taxon caterpillar (internal states in the global scratch), 2 and 23 states."""
    from test_kernel_coverage import _caterpillar
    for S in (2, 23):
        tree, root, _ = _caterpillar(1024, 0.05, 3 + S)
        p = _gpu_problem(S, 4, 1024, 700, tree=(tree, root))
        _kernel_vs_restatement(p, 77, 1)
        p["eng"].close()


@pytest.mark.gpu
def test_c4_shape(gpu_backend):
    """The C4-shaped alignment, 1024 taxa x 131 072 binary columns, GTR + Gamma-4, and two column-offset slices of it
    (cut at a multiple of 64, as a site-sharded run cuts)."""
    from cybayes_b200.engine import Engine
    from large_cases import SEED, _setup
    N, P = 1024, 131072
    aln, codes, _ = _setup(N, P, 2, SEED, 16384)
    tm = [oracle.prob_t("GTR", True, aln.pi, aln.tree, aln.er, r) for r in aln.rates]
    pre = _preorder(aln.tree, aln.root)
    par, ch = [a for a, _ in pre], [b for _, b in pre]
    pool = {i * 4 + k: tm[k][e] for i, e in enumerate(pre) for k in range(4)}
    ps = np.arange(len(pre) * 4, dtype=np.int32).reshape(len(pre), 4)
    mats = np.stack([pool[i] for i in range(len(pre) * 4)])
    seed, rep = 2024, 9

    def run(lo, hi):
        eng = Engine(np.ascontiguousarray(codes[:, lo:hi]), 2, 4)
        eng.alloc_slots(len(pool))
        eng.upload_pmats(np.arange(len(pool), dtype=np.int32), mats)
        out = eng.simulate(par, ch, ps, aln.pi, aln.root, seed, rep, lo)
        eng.close()
        return out
    got = run(0, P)
    want = simulate_restated(codes, 2, 4, par, ch, ps, pool, aln.pi, aln.root, seed, rep)
    assert np.array_equal(got, want)
    cut = 65536 + 64 * 7
    assert np.array_equal(np.concatenate([run(0, cut), run(cut, P)], axis=1), got)


def _golden_state(golden_cases, name):
    import golden_io
    from cybayes_b200 import config
    from cybayes_b200.driver import load_alignment
    case = golden_cases[name]
    load_alignment(golden_io.data_path(case), case["dtype"], case["reader"])
    config.MODEL, config.NORM_BETA = case["model"], case["norm_beta"]
    tree, pi, rates, edges, _ = golden_io.case_state(case)
    return case, tree, pi, rates, edges


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["narrow_F81", "phon_ringe_GTR"])
def test_replicate_lnl_and_statistic(name, golden_cases, gpu_backend):
    """Before the first replicate, the replicate context's lnL of the observed columns is the sample's lnL (the P and
    tree mapping); a replicate's lnL is cb_eval's on a fresh context built from the downloaded replicate, bit for bit,
    and its T is that of the replicate's columns."""
    from cybayes_b200 import config
    from cybayes_b200.alignment import compress_patterns
    from cybayes_b200.engine import Engine
    from cybayes_b200.ML_gamma import matML
    from cybayes_b200.ppc import Replicates, multinomial_statistic
    from cybayes_b200.subst import get_prob_t_all, get_siterates
    case, tree, pi, rates, edges = _golden_state(golden_cases, name)
    srates = 0.8
    site_rates = get_siterates(srates)
    model = case["model"]
    lnl, _ = matML(pi, case["root"], config.LEAF_LLMAT, edges, get_prob_t_all(pi, tree, rates, site_rates),
                   config.N_SITES, config.N_TAXA, config.N_CATS)
    state = {"tree": tree, "root": case["root"], "pi": pi, "rates": rates, "srates": srates, "logLikehood": lnl}
    reps = Replicates(config.LEAF_LLMAT, config.N_CATS)
    assert reps.engine.n_patterns == config.N_SITES
    obs = reps.lnl(state, model)
    assert abs(obs - lnl) <= 1e-12 * abs(lnl), (obs, lnl)
    l_rep, t_rep = reps.draw(state, model, 42, 5)
    assert l_rep != obs
    _, pi_, root, (par, ch, ps), _ = reps._tables(state, model)
    codes = reps.engine.simulate(par, ch, ps, pi_, root, 42, 5)      # the same replicate again: simulation is idempotent
    assert t_rep == multinomial_statistic(compress_patterns(codes)[1])
    fresh = Replicates.__new__(Replicates)
    fresh.engine, fresh.n_cats = Engine(codes, reps.engine.n_states, config.N_CATS, config.LEAF_LLMAT.amb_sets), config.N_CATS
    assert fresh.lnl(state, model) == l_rep
    fresh.close()
    reps.close()


@pytest.mark.gpu
def test_simulate_refuses_a_context_with_a_live_snapshot(gpu_backend):
    from cybayes_b200._lib import CyBayesB200Error
    from cybayes_b200.likelihood import _Plan
    p = _gpu_problem(4, 2, 9, 300)
    eng, tree, root, C = p["eng"], p["tree"], p["root"], p["C"]
    plan = _Plan(oracle.edge_order(tree, root, 9))
    where = {e: i for i, e in enumerate(p["pre"])}
    ps_eval = np.array([p["pslots"][where[e]] for e in plan.edge_keys], dtype=np.int32)
    _, snap = eng.eval(None, plan.nodes, plan.children, ps_eval, p["pi"], want_snapshot=True)
    par, ch = [a for a, _ in p["pre"]], [b for _, b in p["pre"]]
    with pytest.raises(CyBayesB200Error, match="live snapshot"):
        eng.simulate(par, ch, p["pslots"], p["pi"], root, 1, 0)
    eng.release_snapshot(snap)
    with pytest.raises(CyBayesB200Error, match="parents first"):
        eng.simulate(par[::-1], ch[::-1], p["pslots"][::-1], p["pi"], root, 1, 0)
    _kernel_vs_restatement(p, 1, 0)
    eng.close()


@pytest.mark.gpu
def test_drivers_write_the_same_ppc(gpu_backend, tmp_path):
    """narrow.phy F81: .log, .trees and stdout unchanged by --ppc, and the same .ppc from the Python driver and from
    --native."""
    from cybayes_b200 import likelihood
    from cybayes_b200.driver import run_chain
    from cybayes_b200.fastchain import run_chain_native
    py = _runs_with_and_without(run_chain, tmp_path, 600, 50, 3, 17)
    likelihood.reset_engines()
    run_chain_native(NARROW, "F81", 600, 50, "bin", str(tmp_path / "n"), out=io.StringIO(), ppc=3, ppc_seed=17)
    assert open(str(tmp_path / "n.ppc")).read() == py


@pytest.mark.gpu
def test_long_alignment_statistic_takes_the_gpu_route(gpu_backend, monkeypatch):
    """Above the host route's length, T's multiplicities come from cb_compress_patterns without gathering the pattern
    columns: the same weights as the host route."""
    from cybayes_b200 import likelihood
    from cybayes_b200.alignment import compress_patterns
    from cybayes_b200.ppc import column_weights
    rng = np.random.default_rng(5)
    base = rng.integers(0, 3, size=(11, 300)).astype(U8)
    codes = np.ascontiguousarray(base[:, rng.integers(0, 300, size=4000)])
    monkeypatch.setattr(likelihood, "COMPRESS_MAX_SITES", 1000)
    from cybayes_b200 import ppc
    calls = []
    real = ppc.pattern_weights_gpu
    monkeypatch.setattr(ppc, "pattern_weights_gpu", lambda c: calls.append(c.shape) or real(c))
    w = column_weights(codes)
    assert calls == [codes.shape]
    assert np.array_equal(w, compress_patterns(codes)[1])
