"""Every compiled kernel, launched and checked.

launch_ranges picks one kernel instantiation per alignment from the state count, the category count, the pattern
count, the code width and a few knobs.  LEDGER names, for every __global__ instantiation in the library, the case
that launches it; a CPU test holds the ledger equal to what `nm` finds in the binary, so a new instantiation without
a case fails there.  On the GPU each case runs under torch.profiler, which must see its kernel (and no other pruning
kernel of the library), and then through _check_random_inputs: lnL against the scaled oracle, every stored partial,
all schedules bit-equal, dirty paths, batches and device-built P matrices.

Also here: category counts other than 1 and 4 on every multistate family, deep trees whose rate categories need
exponents far apart, the arbitrary-precision pin of the oracle's shared exponent, and the Python surface and both
chain runners at N_CATS != 4."""
import io
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import golden_io
import pruning_oracle as oracle
from conftest import REPO
from test_gpu_parity import _check_random_inputs, _oracle_leaves, _random_problem

CSRC = os.path.join(REPO, "cybayes_b200", "csrc")
LIB = os.path.join(CSRC, "libcybayes_b200.so")
U8, U16 = np.uint8, np.uint16
BIG = 75840   # >= 75 776 patterns: the 256-thread 2-state kernels; 75 840 leaves a ragged last 256- and 512-site block


def kernel_name(demangled):
    """'void cb::prune_s2_kernel<4, 1, 256, 3>(cb::LaunchConst)' -> 'prune_s2_kernel<4, 1, 256, 3>' (None if the
    string names no function)."""
    m = re.search(r"([A-Za-z_]\w*(?:<[^()]*>)?)\(", demangled)
    return m.group(1) if m else None


def _case(kernel, S, C, n_taxa, n_sites, model, dtype=U8, **env):
    return dict(kernel=kernel, S=S, C=C, n_taxa=n_taxa, n_sites=n_sites, model=model, dtype=dtype, env=env)


def _s2t(C, minb, v):
    return _case(f"prune_s2t_kernel<{C}, {minb}, {v}>", 2, C, 20, 700, "F81", CYBAYES_S2_TILED="1",
                 CYBAYES_S2T_MINB=str(minb), CYBAYES_S2T_V=str(v))


def _rc(S, n_taxa=7, n_sites=1060, model="GTR"):
    # 1060 sites: 1088 padded patterns, past the 1 024 where the register-carried kernel takes over, and a ragged
    # last block of 64 of 128 sites
    return _case(f"prune_dmma_rc_kernel<{(S + 7) // 8 * 8}, {'true' if S % 8 == 0 else 'false'}>", S, 4, n_taxa,
                 n_sites, model)


# case id -> the case that launches the kernel; nothing is forced unless the case says so
CASES = {
    # row-major 2-state kernel: 64 threads below 75 776 patterns, 256 threads from there (uint16 codes or tiling off)
    "s2_c4": _case("prune_s2_kernel<4, 1, 64, 8>", 2, 4, 12, 333, "F81"),
    "s2_c1": _case("prune_s2_kernel<1, 1, 64, 8>", 2, 1, 12, 333, "GTR"),
    "s2_big_u16_c4": _case("prune_s2_kernel<4, 1, 256, 3>", 2, 4, 12, BIG, "GTR", U16),
    "s2_big_u16_c1": _case("prune_s2_kernel<1, 1, 256, 4>", 2, 1, 10, BIG, "F81", U16),
    "s2_big_untiled_c4": _case("prune_s2_kernel<4, 1, 256, 3>", 2, 4, 14, BIG, "F81", CYBAYES_S2_TILED="0"),
    "s2_big_untiled_c1": _case("prune_s2_kernel<1, 1, 256, 4>", 2, 1, 16, BIG, "GTR", CYBAYES_S2_TILED="0"),
    "s2_big_minb4_c4": _case("prune_s2_kernel<4, 1, 256, 4>", 2, 4, 11, BIG, "GTR", CYBAYES_S2_TILED="0",
                             CYBAYES_S2_MINB="4"),
    "s2_big_minb4_c1": _case("prune_s2_kernel<1, 1, 256, 4>", 2, 1, 13, BIG, "F81", CYBAYES_S2_TILED="0",
                             CYBAYES_S2_MINB="4"),
    "s2_big_v2_c4": _case("prune_s2_kernel<4, 2, 256, 2>", 2, 4, 12, BIG, "F81", CYBAYES_S2_TILED="0", CYBAYES_S2_V="2"),
    "s2_big_v2_u16_c4": _case("prune_s2_kernel<4, 2, 256, 2>", 2, 4, 15, BIG, "GTR", U16, CYBAYES_S2_V="2"),
    "s2_big_v2_c1": _case("prune_s2_kernel<1, 2, 256, 4>", 2, 1, 10, BIG, "GTR", CYBAYES_S2_TILED="0", CYBAYES_S2_V="2"),
    "s2_big_v2_u16_c1": _case("prune_s2_kernel<1, 2, 256, 4>", 2, 1, 16, BIG, "F81", U16, CYBAYES_S2_V="2"),
    # tiled 2-state kernel <C, resident blocks, tiles per warp>, forced onto a small alignment
    **{f"s2t_c{C}_m{m}_v{v}": _s2t(C, m, v) for C in (4, 1) for m, v in ((3, 2), (2, 2), (2, 1), (3, 1), (4, 1))},
    "general_s7": _case("prune_general_kernel", 7, 4, 9, 200, "GTR"),
    # FP64 tensor-core kernel below 1 024 patterns: compiled state counts, and the run-time one for the rest
    **{f"dmma_s{S}": _case(f"prune_dmma_kernel<{S}>", S, 4, 7, n, m)
       for S, n, m in ((32, 300, "F81"), (40, 90, "GTR"), (47, 64, "GTR"), (48, 129, "GTR"), (56, 200, "JC"),
                       (64, 100, "GTR"))},
    **{f"dmma_s{S}": _case("prune_dmma_kernel<0>", S, 4, 7, n, m)
       for S, n, m in ((33, 70, "GTR"), (45, 130, "F81"), (63, 100, "JC"))},
    # register-carried kernel from 1 024 patterns: <padded S, S == padded S>
    **{f"rc_s{S}": _rc(S) for S in (16, 9, 24, 23, 32, 31, 40, 33, 48, 47, 56, 53, 64, 61)},
}

# pattern compression (cb_compress_patterns): one hash and one verify kernel per code width
COMPRESS_CASES = {"compress_u8": (U8, ["column_hash_kernel<unsigned char>", "column_verify_kernel<unsigned char>"]),
                  "compress_u16": (U16, ["column_hash_kernel<unsigned short>", "column_verify_kernel<unsigned short>"])}

# compiled, but launched by no likelihood path: cb_fp64_peak, the benchmark's FP64 roofline probe
EXEMPT = {"fp64_peak_kernel": "cb_fp64_peak only: the benchmark's FP64 peak probe, no likelihood"}


def helpers(case):
    """The kernels a case launches besides its pruning kernel."""
    fam = case["kernel"].split("<")[0]
    out = {"pmat_build_kernel"}                       # _check_random_inputs builds P matrices on the device
    if fam == "prune_s2t_kernel":
        out.add(f"s2t_image_kernel<{case['C']}>")    # op images, one launch per evaluation
    if fam not in ("prune_s2_kernel", "prune_s2t_kernel"):
        out.add("root_combine_kernel")               # per-category exponents combined at the root
    if fam == "prune_dmma_rc_kernel":
        out.add(f"rc_restage_kernel<{(case['S'] + 7) // 8 * 8}>")
    return out


def _ledger():
    """kernel name -> ids of the cases that launch it."""
    led = {}
    for cid, case in CASES.items():
        for k in {case["kernel"]} | helpers(case):
            led.setdefault(k, []).append(cid)
    for cid, (_, ks) in COMPRESS_CASES.items():
        for k in ks:
            led.setdefault(k, []).append(cid)
    return led


LEDGER = _ledger()
PRUNING = {k for k in LEDGER if k.startswith("prune_")}


# ------------------------------------------------------------------------------------------------ ledger vs binary
def _binary_kernels():
    """Names of the __global__ instantiations in the built library: the host symbols `nm -C` lists under the
    names the sources declare __global__."""
    from cybayes_b200 import _lib
    _lib.load()                                       # raises if the library is not built
    nm = shutil.which("nm")
    if nm is None:
        pytest.skip("nm unavailable")
    src = "".join(open(os.path.join(CSRC, f)).read() for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh")))
    declared = set(re.findall(r"__global__\s+void\s+(?:__launch_bounds__\([^)]*\)\s+)?(\w+)\s*\(", src))
    assert len(declared) >= 12, declared
    out = subprocess.run([nm, "-C", "--defined-only", LIB], capture_output=True, text=True, check=True).stdout
    found = set()
    for line in out.splitlines():
        parts = line.split(None, 2)
        if len(parts) < 3 or parts[1] not in "TtWw" or "__device_stub__" in parts[2]:
            continue
        name = kernel_name(parts[2])
        if name and name.split("<")[0] in declared:
            found.add(name)
    assert {n.split("<")[0] for n in found} == declared, "a __global__ declared in the sources is not in the binary"
    return found


def test_ledger_names_every_kernel_in_the_binary():
    """Every instantiation nm finds has a case (or is an explained exemption), and every ledger entry exists."""
    found = _binary_kernels()
    listed = set(LEDGER) | set(EXEMPT)
    assert not set(LEDGER) & set(EXEMPT)
    assert not found - listed, f"kernels without a test case: {sorted(found - listed)}"
    assert not listed - found, f"ledger entries the binary does not contain: {sorted(listed - found)}"
    assert len(found) >= 55


def test_ledger_cases_select_their_kernel_by_shape():
    """The ledger's cases reach the parts of launch_ranges they are meant to: what decides the kernel is the shape."""
    for cid, c in CASES.items():
        P = -(-c["n_sites"] // 64) * 64
        fam = c["kernel"].split("<")[0]
        if fam == "prune_s2_kernel":
            assert (P >= 75776) == ("256" in c["kernel"]), cid
            if P >= 75776:
                assert c["dtype"] is U16 or c["env"].get("CYBAYES_S2_TILED") == "0", cid
        elif fam == "prune_dmma_kernel":
            assert 32 <= c["S"] <= 64 and P < 1024 and not c["env"], cid
        elif fam == "prune_dmma_rc_kernel":
            assert 9 <= c["S"] <= 64 and P >= 1024 and P % 128 == 64 and not c["env"], cid
    big = [c for c in CASES.values() if c["n_sites"] == BIG]
    assert {c["C"] for c in big} == {1, 4} and all(10 <= c["n_taxa"] <= 16 for c in big)


# ------------------------------------------------------------------------------------------- run and prove on GPU
def launched_kernels(fn):
    """Run fn() under torch.profiler (CUDA activities); the library's kernel names the profiler recorded."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {kernel_name(e.name) for e in prof.events() if e.device_type == DeviceType.CUDA}
    return names & (set(LEDGER) | set(EXEMPT))


def _run_case(case, monkeypatch):
    for k, v in case["env"].items():
        monkeypatch.setenv(k, v)
    got = launched_kernels(lambda: _check_random_inputs(case["S"], case["n_taxa"], case["n_sites"], case["model"],
                                                        n_cats=case["C"], code_dtype=case["dtype"]))
    want = {case["kernel"]} | helpers(case)
    assert got == want, f"expected {sorted(want)}, the profiler saw {sorted(got)}"
    print(f"launched: {sorted(got)}")


@pytest.mark.gpu
@pytest.mark.parametrize("cid", list(CASES))
def test_ledger_case(cid, gpu_backend, monkeypatch):
    _run_case(CASES[cid], monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("cid", list(COMPRESS_CASES))
def test_ledger_compression_case(cid, gpu_backend):
    """cb_compress_patterns with 1- and 2-byte codes: the same result as the host route, element for element."""
    from cybayes_b200.alignment import compress_patterns, compress_patterns_gpu
    dtype, kernels = COMPRESS_CASES[cid]
    rng = np.random.default_rng(31)
    base = rng.integers(0, 300 if dtype is U16 else 30, size=(9, 400)).astype(dtype)
    codes = np.ascontiguousarray(base[:, rng.integers(0, base.shape[1], size=5000)])
    codes[rng.integers(0, 9, size=500), rng.integers(0, 5000, size=500)] ^= 1
    out = []
    got = launched_kernels(lambda: out.append(compress_patterns_gpu(codes)))
    assert got == set(kernels), got
    p0, w0, m0 = compress_patterns(codes)
    p1, w1, m1 = out[0]
    assert p1.dtype == dtype and np.array_equal(p0, p1) and np.array_equal(w0, w1) and np.array_equal(m0, m1)
    assert w1.sum() == codes.shape[1] and np.array_equal(p1[:, m1], codes)


# ----------------------------------------------------------------------------------------- category-count sweep
# The rates are those of site_rates / get_siterates, restated from the reference: for C = 3, 6 and 7 its
# np.arange(1/C, 1, 1/C) yields a last quantile point at 1.0, so the last category gets rate 0 (an identity P).
# The categories still differ from one another, which is what these tests need.
SWEEP = {   # family -> (S, taxa, sites, model, code dtype, kernel for C = 1, kernel otherwise)
    "binary_general": (2, 12, 333, "F81", U8, "prune_s2_kernel<1, 1, 64, 8>", "prune_general_kernel"),
    "general_s7": (7, 9, 200, "GTR", U8, "prune_general_kernel", "prune_general_kernel"),
    "general_s130_u16": (130, 6, 129, "F81", U16, "prune_general_kernel", "prune_general_kernel"),
    "dmma_s45": (45, 8, 130, "GTR", U8, "prune_dmma_kernel<0>", "prune_dmma_kernel<0>"),
    "dmma_s48": (48, 6, 129, "GTR", U8, "prune_dmma_kernel<48>", "prune_dmma_kernel<48>"),
    "rc_s24": (24, 7, 1060, "GTR", U8, "prune_dmma_rc_kernel<24, true>", "prune_dmma_rc_kernel<24, true>"),
    "rc_s64": (64, 7, 1060, "F81", U8, "prune_dmma_rc_kernel<64, true>", "prune_dmma_rc_kernel<64, true>"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("n_cats", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("family", list(SWEEP))
def test_category_count(family, n_cats, gpu_backend, monkeypatch):
    """C = 1 .. 8 (CB_MAX_CATS) on every family that takes it, each category with its own rate."""
    S, n_taxa, n_sites, model, dtype, k1, k = SWEEP[family]
    _run_case(_case(k1 if n_cats == 1 else k, S, n_cats, n_taxa, n_sites, model, dtype), monkeypatch)


def test_random_problem_gives_each_category_its_rate():
    for C in (2, 3, 5, 8):
        rates = _random_problem(1, 4, 10, 3, n_cats=C)[-1]
        assert len(rates) == C and len(set(rates)) == C, rates
    assert _random_problem(1, 4, 10, 3, n_cats=1)[-1] == [1.0]
    assert _random_problem(1, 4, 10, 2, code_dtype=U16)[3].dtype == U16


@pytest.mark.gpu
def test_nine_categories_are_rejected(gpu_backend):
    from cybayes_b200._lib import CyBayesB200Error
    from cybayes_b200.engine import Engine
    with pytest.raises(CyBayesB200Error, match=r"n_cats must be 1\.\.8"):
        Engine(np.zeros((3, 8), dtype=U8), 7, 9)


# ---------------------------------------------------------------------------- deep trees, categories far apart
ALPHA_DEEP = 0.05


def _caterpillar(n_taxa, bl_mean, seed):
    rng = np.random.default_rng(seed)
    tree, prev, nxt = {}, 1, n_taxa + 1
    for tip in range(2, n_taxa + 1):
        tree[nxt, prev] = float(rng.exponential(bl_mean))
        tree[nxt, tip] = float(rng.exponential(bl_mean))
        prev, nxt = nxt, nxt + 1
    return tree, nxt - 1, rng


DEEP = {   # family -> (S, sites, model, kernel)
    "general": (7, 96, "GTR", "prune_general_kernel"),
    "dmma": (40, 100, "F81", "prune_dmma_kernel<40>"),
    "dmma_rc": (24, 1060, "F81", "prune_dmma_rc_kernel<24, true>"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(DEEP))
def test_deep_tree_with_categories_far_apart(family, gpu_backend):
    """A 400-taxon caterpillar with long branches and alpha = 0.05: the unscaled pruning underflows, and the
    per-category exponents of these kernels drift far apart (root_combine_kernel adds categories whose exponents
    differ by many binades).  lnL against the scaled oracle; a dirty path gives the same bits."""
    from cybayes_b200.engine import Engine
    from cybayes_b200.likelihood import _Plan
    S, n_sites, model, kernel = DEEP[family]
    n_taxa, C = 400, 4
    tree, root, rng = _caterpillar(n_taxa, 0.6, 11 + S)
    edges = oracle.edge_order(tree, root, n_taxa)
    codes = rng.integers(0, S, size=(n_taxa, n_sites))
    codes[rng.random((n_taxa, n_sites)) < 0.05] = S
    codes = codes.astype(U8)
    pi = rng.dirichlet(np.full(S, 5.0))
    er = rng.dirichlet(np.ones(S * (S - 1) // 2))
    rates = oracle.site_rates(ALPHA_DEEP, C)
    tm = [oracle.prob_t(model, False, pi, tree, er, r) for r in rates]
    leaves = _oracle_leaves(codes, S, np.ones((1, S)))
    assert oracle.mat_ml(pi, root, leaves, edges, tm, n_sites, n_taxa, n_cats=C)[0] == -np.inf
    want = oracle.mat_ml_scaled(pi, root, leaves, edges, tm, n_sites, n_taxa, n_cats=C)
    res = {}

    def run():
        eng = Engine(codes, S, C)
        plan = _Plan(edges)
        ekeys = list(tree)
        block = eng.alloc_slots(len(ekeys) * C)
        slot_of = {(k, e): block.base + k * len(ekeys) + i for k in range(C) for i, e in enumerate(ekeys)}
        eng.upload_pmats(np.arange(block.base, block.base + block.n, dtype=np.int32),
                         np.stack([tm[k][e] for k in range(C) for e in ekeys]))
        pslots = np.array([[slot_of[k, e] for k in range(C)] for e in plan.edge_keys], dtype=np.int32)
        res["lnl"], snap = eng.eval(None, plan.nodes, plan.children, pslots, pi)
        path = sorted(oracle.path_to_root(oracle.parent_of(tree), 40, root), key=plan.index.__getitem__)
        ch = np.array([c for n in path for c in plan.kids[n]], dtype=np.int32)
        ps = np.array([[slot_of[k, (n, c)] for k in range(C)] for n in path for c in plan.kids[n]], dtype=np.int32)
        res["dirty"], _ = eng.eval(snap, np.array(path, dtype=np.int32), ch, ps, pi, want_snapshot=False)
        eng.release_snapshot(snap)
        eng.close()
    got = launched_kernels(run)
    assert kernel in got and not (got & PRUNING) - {kernel}, got
    assert np.isfinite(res["lnl"]) and abs(res["lnl"] - want) <= 1e-12 * abs(want), (res["lnl"], want)
    assert res["dirty"] == res["lnl"]


def _mp_lnl(pi, root, leaves, edges, tm, n_sites, n_taxa, C):
    """The unscaled pruning pass of mat_ml restated in 50-digit arithmetic on the same (exactly converted) P
    matrices: no underflow, no rescaling, nothing shared between categories."""
    import mpmath
    mp = mpmath.mp
    S = len(pi)
    total = [mp.mpf(0)] * n_sites
    for k in range(C):
        part = {}
        for parent, child in edges:
            P = [[mp.mpf(float(x)) for x in row] for row in tm[k][parent, child]]
            if child <= n_taxa:
                src = [[mp.mpf(float(x)) for x in row] for row in leaves[child]]
            else:
                src = part.pop(child)
            v = [[mp.fsum(P[i][j] * src[j][p] for j in range(S) if src[j][p]) for p in range(n_sites)]
                 for i in range(S)]
            if parent in part:
                v = [[a * b for a, b in zip(ra, rb)] for ra, rb in zip(part[parent], v)]
            part[parent] = v
        for p in range(n_sites):
            total[p] += mp.fsum(mp.mpf(float(pi[i])) * part[root][i][p] for i in range(S)) / C
    return mp.fsum(mp.log(t) for t in total)


@pytest.mark.parametrize("S", [3, 24])
def test_shared_exponent_oracle_matches_arbitrary_precision(S):
    """mat_ml_scaled keeps one power-of-two exponent per site for all categories; the GPU families keep one per
    category.  Pin the oracle once against exact arithmetic where the categories are far apart (alpha = 0.05, long
    branches): the deep-tree tests above then compare the kernels with a checked reference."""
    import mpmath
    n_taxa, n_sites, C = 40, 8, 4
    tree, root, rng = _caterpillar(n_taxa, 0.6, 5 + S)
    edges = oracle.edge_order(tree, root, n_taxa)
    codes = rng.integers(0, S + 1, size=(n_taxa, n_sites)).astype(U8)
    pi = rng.dirichlet(np.full(S, 5.0))
    rates = oracle.site_rates(ALPHA_DEEP, C)
    assert rates[-1] / rates[0] > 1e6
    tm = [oracle.prob_t("F81", False, pi, tree, None, r) for r in rates]
    leaves = _oracle_leaves(codes, S, np.ones((1, S)))
    want = oracle.mat_ml_scaled(pi, root, leaves, edges, tm, n_sites, n_taxa, n_cats=C)
    saved = mpmath.mp.dps
    mpmath.mp.dps = 50
    try:
        exact = _mp_lnl(pi, root, leaves, edges, tm, n_sites, n_taxa, C)
    finally:
        mpmath.mp.dps = saved
    assert abs(want - float(exact)) <= 1e-13 * abs(float(exact)), (want, exact)


# -------------------------------------------------------------------------- Python surface and chains, C != 4
def _surface_check(name, n_cats, golden_cases, monkeypatch):
    from cybayes_b200 import config
    from cybayes_b200.driver import load_alignment
    from cybayes_b200.mcmc_gamma import (adjlist2reverse_nodes_dict, get_edge_transition_mat, get_path2root,
                                         get_prob_t)
    from cybayes_b200.ML_gamma import cache_matML, matML
    from cybayes_b200.subst import get_siterates
    case = golden_cases[name]
    monkeypatch.setattr(config, "N_CATS", n_cats)
    load_alignment(golden_io.data_path(case), case["dtype"], case["reader"])
    config.MODEL, config.NORM_BETA = case["model"], case["norm_beta"]
    tree, pi, rates, edges, _ = golden_io.case_state(case)
    if rates is None:   # not stored for models that do not use exchangeabilities
        rates = np.ones(1)
    site_rates = get_siterates(0.37)
    assert len(site_rates) == n_cats
    root, N = case["root"], case["n_taxa"]
    args = (config.N_SITES, config.N_TAXA, n_cats)
    _, _, _, _, ll, _, n_sites = oracle.read_phylip(golden_io.data_path(case), case["reader"])
    rel = 1e-9 if case["model"] == "GTR" else 1e-11

    def oracle_tm(t):
        return [oracle.prob_t(case["model"], case["dtype"] == "bin", pi, t, rates, r, beta=case["norm_beta"])
                for r in site_rates]
    tmats = [get_prob_t(pi, tree, rates, r) for r in site_rates]
    lnl, cache = matML(pi, root, config.LEAF_LLMAT, edges, tmats, *args)
    want, want_cache = oracle.mat_ml(pi, root, ll, edges, oracle_tm(tree), n_sites, N, n_cats=n_cats)
    assert abs(lnl - want) <= rel * abs(want), (lnl, want)
    for node in sorted(want_cache[0])[::7]:
        if node != root:
            ref = np.stack([want_cache[k][node] for k in range(n_cats)])
            # GTR: eigendecomposition against expm, so the smallest entries of P agree to an absolute error only
            np.testing.assert_allclose(cache.partial(node), ref, rtol=rel * 10,
                                       atol=1e-14 if case["model"] == "GTR" else 0)
    e = next(k for k in tree if k[1] <= N)
    tree2 = dict(tree)
    tree2[e] = tree[e] * 1.7
    for k, r in enumerate(site_rates):
        tmats[k][e] = get_edge_transition_mat(pi, rates, tree2[e] * r)
    path = get_path2root(adjlist2reverse_nodes_dict(tree), e[1], root)
    l2, _ = cache_matML(pi, root, config.LEAF_LLMAT, cache, path, edges, tmats, *args)
    want2 = oracle.mat_ml(pi, root, ll, edges, oracle_tm(tree2), n_sites, N, n_cats=n_cats)[0]
    assert abs(l2 - want2) <= rel * abs(want2) and l2 != lnl, (l2, want2)


@pytest.mark.gpu
@pytest.mark.parametrize("n_cats", [3, 8])
@pytest.mark.parametrize("name", ["phon_ringe_GTR", "ielex_multistate_F81"])
def test_python_surface_category_count(name, n_cats, golden_cases, gpu_backend, monkeypatch):
    """ML_gamma.matML and cache_matML with config.N_CATS = 3 and 8: lnL and partials against the oracle."""
    _surface_check(name, n_cats, golden_cases, monkeypatch)


def _driver_vs_native(backend, tmp_path, monkeypatch, n_gen):
    """The Python driver and the native generation loop at N_CATS = 3: the same move, proposal lnL and decision in
    every generation, and the same sampled trees."""
    from cybayes_b200 import config
    from cybayes_b200.driver import run_chain
    from cybayes_b200.fastchain import run_chain_native
    monkeypatch.setattr(config, "N_CATS", 3)
    path = os.path.join(REPO, "tests", "golden", "data", "phon_ringe.phy")
    a, b = [], []
    ra = run_chain(path, "F81", n_gen, 10, "multi", str(tmp_path / "d"), out=io.StringIO(), fast_spr=True,
                   on_generation=lambda i, cur, prop, p, mv, acc, st: a.append((p, mv, acc, float(prop))))
    backend.reset_engines()
    rb = run_chain_native(path, "F81", n_gen, 10, "multi", str(tmp_path / "n"), out=io.StringIO(),
                          on_generation=lambda i, cur, prop, p, mv, acc, st: b.append((p, mv, acc, float(prop))))
    assert len(a) == n_gen and len(b) == n_gen
    assert [x[:3] for x in a] == [x[:3] for x in b]
    np.testing.assert_allclose([x[3] for x in a], [x[3] for x in b], rtol=1e-12)
    assert sum(x[2] for x in a) > 10 and len({x[0] for x in a}) >= 3
    assert abs(ra["initial_lnL"] - rb["initial_lnL"]) <= 1e-12 * abs(ra["initial_lnL"])
    assert open(str(tmp_path / "d.trees")).read() == open(str(tmp_path / "n.trees")).read()


@pytest.mark.gpu
def test_driver_and_native_chain_agree_with_three_categories(gpu_backend, tmp_path, monkeypatch):
    _driver_vs_native(gpu_backend, tmp_path, monkeypatch, 300)


def test_driver_and_native_chain_agree_with_three_categories_on_the_fake_engine(fake_backend, tmp_path, monkeypatch):
    from cybayes_b200 import likelihood
    _driver_vs_native(likelihood, tmp_path, monkeypatch, 300)
