"""Snapshot lineages on the 2-state kernels, pattern weights on every kernel family, recorded chain traces on the tiled
2-state kernel.

1. A seeded chain of proposals (branch length, NNI, external SPR, pi / alpha) drives `Engine` the way an MCMC loop does:
   every dirty path starts from the snapshot of the previous accepted state, accepted proposals release their parent
   while the child still shares its records, and a reservoir of old snapshots (retain_snapshot) is revisited with new
   dirty paths.  Every P slot an evaluation does not reference holds NaN matrices, so a record that reads a P matrix
   after its slot was reused turns lnL into NaN.  Every dirty-path lnL must equal a fresh full pass bit for bit, kept
   partials and records must equal a fresh full pass's (mantissas and exponents), and lnL must equal the scaled oracle
   with the same weights.  The same lineage function also runs, unmarked, on the oracle-backed fake engine.
2. Random non-unit pattern weights (zeros included) on each kernel family, against the weighted oracle; compressed
   patterns with multiplicities against the uncompressed alignment on the tiled kernel.
3. The recorded binary chain traces, both runners, with the tiled kernel forced on."""
import numpy as np
import pytest

import pruning_oracle as oracle
from test_gpu_parity import _oracle_leaves, _random_problem
from test_gpu_parity import test_c1_at_its_stated_length as _c1_at_its_stated_length
from test_gpu_parity import test_driver_trace_matches_reference as _driver_trace
from test_gpu_parity import test_native_chain_trace_matches_reference as _native_trace
from trace_checks import TRACES

KERNEL_ENV = ("CYBAYES_S2_TILED", "CYBAYES_S2T_V", "CYBAYES_S2T_MINB", "CYBAYES_S2T_SLOTS", "CYBAYES_S2T_BULK",
              "CYBAYES_S2T_SMALL_RECS", "CYBAYES_DMMA_RC", "CYBAYES_RC_MIN_STATES", "CYBAYES_CHAIN_LNL_FIRST")


def _set_env(monkeypatch, env):
    for k in KERNEL_ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def _weights(rng, n):
    """Integer pattern multiplicities: mostly small, some up to 1000, about one in ten zero."""
    w = rng.integers(1, 8, size=n).astype(np.float64)
    big = rng.random(n) < 0.05
    w[big] = rng.integers(100, 1001, size=int(big.sum()))
    w[rng.random(n) < 0.1] = 0.0
    return w


# ---------------------------------------------------------------------------------------------------------- lineage
class _State:
    """One chain state: tree (edge -> length), pi, category rates and the P-slot group of every edge."""
    __slots__ = ("tree", "pi", "rates", "groups", "plan", "parents")

    def __init__(self, tree, pi, rates, groups, root, n_taxa, like=None):
        from cybayes_b200.likelihood import _Plan
        self.tree, self.pi, self.rates, self.groups = tree, pi, rates, groups
        if like is not None:     # same topology
            self.plan, self.parents = like.plan, like.parents
        else:
            self.plan = _Plan(oracle.edge_order(tree, root, n_taxa))
            self.parents = oracle.parent_of(tree)


def run_lineage(make_engine, n_taxa, n_sites, n_cats, n_gen, seed, reservoir, check_every=25, pull_every=6):
    """Run a seeded chain of `n_gen` proposals on a random tree; returns every lnL the chain computed, in order, and
    the peak number of folded-cherry records held by live snapshots.  Accept / reject decisions, moves and reservoir
    choices come from the seed alone, so any two engines see the same sequence of op lists."""
    from cybayes_b200.driver import _spr_dirty_nodes
    rng = np.random.default_rng(seed)
    tree0, root, _, codes, amb, pi0, _, _ = _random_problem(seed, n_taxa, n_sites, 2, n_cats=n_cats)
    N, C = n_taxa, n_cats
    w = _weights(rng, n_sites)
    leaves = _oracle_leaves(codes, 2, amb)
    eng = make_engine(codes, 2, C, amb, w)
    has_info = hasattr(eng, "last_eval_info")

    # P slots: groups of C consecutive slots, one group per (edge, state); a changed edge always gets a group no live
    # state uses, taken lowest index first so freed groups are reused soon
    n_edges = 2 * N - 2
    G = (reservoir + 4) * n_edges
    block = eng.alloc_slots(G * C)
    host = np.full((G, C, 2, 2), np.nan)
    dev_ok = np.zeros(G, bool)     # the device holds host[g]
    dev_nan = np.zeros(G, bool)    # the device holds NaN matrices
    free = []

    def alloc(mats):
        g = free.pop()
        host[g] = mats
        dev_ok[g] = False
        return g

    def pmats(pi, rates, bl):
        return np.stack([oracle.prob_t("F81", True, pi, {(0, 0): bl}, None, r)[0, 0] for r in rates])

    def rates_of(alpha):
        return oracle.site_rates(alpha, C) if C == 4 else [1.0]

    def ops(st, nodes):
        kids = st.plan.kids
        ch = np.array([c for n in nodes for c in kids[n]], dtype=np.int32)
        gs = np.array([st.groups[n, c] for n in nodes for c in kids[n]], dtype=np.int64)
        ps = (block.base + gs[:, None] * C + np.arange(C)[None, :]).astype(np.int32)
        return np.array(nodes, dtype=np.int32), ch, ps, gs

    def full(st):
        return ops(st, st.plan.node_list)

    def dirty(st, dset):
        return ops(st, sorted(set(dset), key=st.plan.index.__getitem__))

    # host model of the folded-cherry records each snapshot holds: {cherry node: record id}; a dirty path replaces the
    # records of the nodes it recomputes and shares every other record with its input snapshot
    recs, refc, next_rec, peak = {}, {}, [0], [0]

    def run(snap_in, st, op, want):
        nodes, ch, ps, gs = op
        ref = np.zeros(G, bool)
        ref[gs] = True
        up = np.nonzero((ref & ~dev_ok) | (~ref & ~dev_nan))[0]
        if up.size:
            mats = np.where(ref[up][:, None, None, None], host[up], np.nan)
            slots = (block.base + up[:, None] * C + np.arange(C)[None, :]).astype(np.int32).ravel()
            eng.upload_pmats(slots, mats.reshape(-1, 2, 2))
            dev_ok[up], dev_nan[up] = ref[up], ~ref[up]
        # the single-launch walk, which large alignments take by default: it keeps small subtrees as records
        lnl, sid = eng.eval(snap_in, nodes, ch, ps, st.pi, want_snapshot=want, force_walk=True)
        assert np.isfinite(lnl), (lnl, "a P slot that was poisoned has been read")
        in_list = set(nodes.tolist())
        made = []
        for i, n in enumerate(nodes.tolist()):
            a, b = st.plan.kids[n]
            if a <= N and b <= N and i != len(nodes) - 1 and st.parents[n] in in_list:
                made.append(n)
        if has_info:
            assert eng.last_eval_info()["cherries_folded"] == len(made)
        if want:
            held = dict(recs[snap_in]) if snap_in is not None else {}
            for n in in_list:
                held.pop(n, None)
            for n in made:
                held[n] = next_rec[0]
                next_rec[0] += 1
            recs[sid], refc[sid] = held, 1
        return lnl, (sid if want else -1)

    def retain(s):
        eng.retain_snapshot(s)
        refc[s] += 1

    def release(s):
        eng.release_snapshot(s)
        refc[s] -= 1
        if refc[s] == 0:
            del recs[s], refc[s]

    def count_live():
        peak[0] = max(peak[0], len({r for s in recs for r in recs[s].values()}))

    def propose(st, kind):
        tree, groups = dict(st.tree), dict(st.groups)
        keys = list(tree)
        if kind == "spr":
            for _ in range(200):
                leaf = int(rng.integers(1, N + 1))
                hub = st.parents[leaf]
                tgt = keys[int(rng.integers(len(keys)))]
                if not (hub == root or hub in tgt or st.parents[hub] in tgt):
                    break
            else:
                kind = "bl"
        if kind == "bl":
            tip_edge = rng.random() < 0.5
            pool = [e for e in keys if (e[1] <= N) == tip_edge]
            e = pool[int(rng.integers(len(pool)))]
            tree[e] = tree[e] * float(np.exp(rng.uniform(-0.7, 0.7)))
            groups[e] = alloc(pmats(st.pi, st.rates, tree[e]))
            return _State(tree, st.pi, st.rates, groups, root, N, like=st), oracle.path_to_root(st.parents, e[1], root)
        if kind == "nni":
            inner = [e for e in keys if e[1] > N]
            a, b = inner[int(rng.integers(len(inner)))]
            ka, kb = st.plan.kids[a], st.plan.kids[b]
            src = ka[0] if ka[1] == b else ka[1]
            tgt = kb[int(rng.integers(2))]
            sbl, tbl = tree.pop((a, src)), tree.pop((b, tgt))
            del groups[a, src], groups[b, tgt]
            tree[a, tgt], tree[b, src] = tbl, sbl
            groups[a, tgt], groups[b, src] = alloc(pmats(st.pi, st.rates, tbl)), alloc(pmats(st.pi, st.rates, sbl))
            new = _State(tree, st.pi, st.rates, groups, root, N)
            return new, [b] + oracle.path_to_root(new.parents, b, root)
        if kind == "spr":   # prune `leaf` with its parent, regraft on `tgt` (moves.externalSPR)
            up = st.parents[hub]
            other = [c for c in st.plan.kids[hub] if c != leaf][0]
            x, y, r = tree.pop((up, hub)), tree.pop((hub, other)), tree.pop(tgt)
            for e in ((up, hub), (hub, other), tgt):
                del groups[e]
            u = float(rng.uniform(0.05, 0.95))
            tree[tgt[0], hub], tree[hub, tgt[1]], tree[up, other] = r * u, r * (1.0 - u), x + y
            for e in ((tgt[0], hub), (hub, tgt[1]), (up, other)):
                groups[e] = alloc(pmats(st.pi, st.rates, tree[e]))
            return _State(tree, st.pi, st.rates, groups, root, N), _spr_dirty_nodes(st.parents, tree, root)
        # pi and alpha: every matrix changes, a full pass
        pi = rng.dirichlet(200.0 * st.pi)
        rates = rates_of(float(rng.uniform(0.3, 2.0)))
        groups = {e: alloc(pmats(pi, rates, bl)) for e, bl in tree.items()}
        return _State(tree, pi, rates, groups, root, N, like=st), None

    def fresh_equal(st, lnl):
        """check 1: a fresh full pass of the state gives the same bits"""
        got, _ = run(None, st, full(st), False)
        assert got == lnl, (got, lnl)

    def same_partials(st, s, lnl):
        """check 2: every kept partial and record of snapshot s equals a fresh full pass's, mantissas and exponents"""
        got, s_f = run(None, st, full(st), True)
        assert got == lnl, (got, lnl)
        for n in st.plan.node_list[:-1]:
            a, ea = eng.read_partial(s, n, with_scale=True)
            b, eb = eng.read_partial(s_f, n, with_scale=True)
            assert np.array_equal(a, b) and np.array_equal(ea, eb), n
        release(s_f)

    def oracle_equal(st, lnl):
        """check 3: the scaled oracle on the same host matrices and weights"""
        tm = [{e: host[g][k] for e, g in st.groups.items()} for k in range(C)]
        want = oracle.mat_ml_scaled(st.pi, root, leaves, st.plan.edges, tm, n_sites, N, n_cats=C, weights=w)
        assert abs(lnl - want) <= 1e-12 * abs(want), (lnl, want)

    def refill_free(states):
        used = set()
        for st in states:
            used.update(st.groups.values())
        free[:] = sorted(set(range(G)) - used, reverse=True)

    refill_free([])
    rates0 = rates_of(0.7)
    cur = _State(dict(tree0), pi0, rates0, {e: alloc(pmats(pi0, rates0, bl)) for e, bl in tree0.items()}, root, N)
    cur_lnl, cur_snap = run(None, cur, full(cur), True)
    oracle_equal(cur, cur_lnl)
    trace = [cur_lnl]
    res = []    # reservoir: [state, snapshot, lnL]

    def keep(st, s, lnl):
        retain(s)
        res.append([st, s, lnl])
        if len(res) > reservoir:
            release(res.pop(0)[1])
        count_live()

    for gen in range(1, n_gen + 1):
        refill_free([cur] + [r[0] for r in res])
        kind = ("bl", "nni", "spr", "model")[int(rng.choice(4, p=[0.4, 0.2, 0.15, 0.25]))]
        prop, dset = propose(cur, kind)
        lnl_first = dset is None and rng.random() < 0.5
        if dset is None:
            lnl_p, snap_p = run(None, prop, full(prop), not lnl_first)
        else:
            lnl_p, snap_p = run(cur_snap, prop, dirty(prop, dset), True)
            fresh_equal(prop, lnl_p)
        trace.append(lnl_p)
        count_live()
        if rng.random() < 0.5:       # accept
            if lnl_first:           # likelihood first: repeat keeping the cache
                again, snap_p = run(None, prop, full(prop), True)
                assert again == lnl_p
            release(cur_snap)       # the child may still share the parent's records
            cur, cur_snap, cur_lnl = prop, snap_p, lnl_p
            if dset is None or rng.random() < 0.1:
                keep(cur, cur_snap, cur_lnl)
        elif snap_p >= 0:
            if dset is None or rng.random() < 0.1:
                keep(prop, snap_p, lnl_p)
            release(snap_p)
        if res and gen % pull_every == 0:
            # an old snapshot: its partials first, then a dirty path from it with the state it was made with
            i = int(rng.integers(len(res)))
            st_r, s_r, l_r = res[i]
            same_partials(st_r, s_r, l_r)
            child, dset = propose(st_r, ("bl", "nni", "spr")[int(rng.integers(3))])
            l_c, s_c = run(s_r, child, dirty(child, dset), True)
            fresh_equal(child, l_c)
            trace.append(l_c)
            count_live()
            if rng.random() < 0.5:   # the child replaces its parent, which goes while the child shares its records
                res[i] = [child, s_c, l_c]
                release(s_r)
            else:
                release(s_c)
        if gen % check_every == 0 or gen == n_gen:
            same_partials(cur, cur_snap, cur_lnl)
            oracle_equal(cur, cur_lnl)

    release(cur_snap)
    for r in res:
        release(r[1])
    assert not recs and not refc
    if hasattr(eng, "stats"):   # check 4: nothing leaked (buffers, records)
        before = eng.stats()["device_bytes"]
        a, s_a = run(None, cur, full(cur), True)
        b, s_b = run(None, cur, full(cur), True)
        release(s_a)
        release(s_b)
        assert a == b == cur_lnl
        assert eng.stats()["device_bytes"] == before
    eng.close()
    return trace, peak[0]


class _RefCountedFake:
    """tests/fake_engine.FakeEngine with the library's snapshot lifetime: retain / release count holders."""

    def __new__(cls, codes, n_states, n_cats, amb_sets=None, weights=None):
        from fake_engine import FakeEngine

        class Fake(FakeEngine):
            def eval(self, snapshot, *a, **kw):
                assert snapshot is None or self.refs.get(snapshot, 0) > 0, snapshot
                lnl, sid = super().eval(snapshot, *a, **kw)
                if sid >= 0:
                    self.refs[sid] = 1
                return lnl, sid

            def retain_snapshot(self, s):
                assert self.refs.get(s, 0) > 0
                self.refs[s] += 1

            def release_snapshot(self, s):
                assert self.refs.get(s, 0) > 0
                self.refs[s] -= 1
                if self.refs[s] == 0:
                    del self.refs[s], self.snaps[s]

            def read_partial(self, snap, node, with_scale=False):
                assert self.refs.get(snap, 0) > 0
                return super().read_partial(snap, node, with_scale)

        eng = Fake(codes, n_states, n_cats, amb_sets, weights)
        eng.refs = {}
        return eng


def test_lineage_driver_dry_run_on_the_fake_engine():
    """The lineage driver's own logic (moves, op lists, slot poisoning, reservoir, snapshot lifetimes) on CPU."""
    trace, peak = run_lineage(_RefCountedFake, 24, 150, 4, 30, 7, reservoir=4, check_every=10, pull_every=3)
    assert len(trace) > 1 + 30 and all(np.isfinite(trace)) and peak > 0
    trace1, _ = run_lineage(_RefCountedFake, 17, 70, 1, 12, 8, reservoir=3, check_every=5, pull_every=4)
    assert len(trace1) > 1 + 12


LINEAGE_ENV = {
    "row": {"CYBAYES_S2_TILED": "0"},
    "tiled": {"CYBAYES_S2_TILED": "1"},
    "tiled_v1_minb4_slots1": {"CYBAYES_S2_TILED": "1", "CYBAYES_S2T_V": "1", "CYBAYES_S2T_MINB": "4",
                              "CYBAYES_S2T_SLOTS": "1"},
    "tiled_spills": {"CYBAYES_S2_TILED": "1", "CYBAYES_S2T_SLOTS": "0"},
    "tiled_bulk": {"CYBAYES_S2_TILED": "1", "CYBAYES_S2T_BULK": "1"},
    "tiled_no_small_recs": {"CYBAYES_S2_TILED": "1", "CYBAYES_S2T_SMALL_RECS": "0"},
}
LINEAGE = [("row", 4), ("row", 1), ("tiled", 4), ("tiled", 1), ("tiled_v1_minb4_slots1", 4), ("tiled_spills", 4),
           ("tiled_bulk", 4), ("tiled_no_small_recs", 4)]
LINEAGE_SHAPE = {4: (240, 1237, 200, 31), 1: (300, 2999, 160, 32)}   # taxa, patterns, generations, seed
LINEAGE_RESERVOIR = 20
_sequences = {}


def _engine(codes, n_states, n_cats, amb, weights):
    from cybayes_b200.engine import Engine
    return Engine(codes, n_states, n_cats, amb, weights=weights)


def _lineage(name, n_cats, monkeypatch):
    if (name, n_cats) not in _sequences:
        _set_env(monkeypatch, LINEAGE_ENV[name])
        n_taxa, n_sites, n_gen, seed = LINEAGE_SHAPE[n_cats]
        trace, peak = run_lineage(_engine, n_taxa, n_sites, n_cats, n_gen, seed, LINEAGE_RESERVOIR)
        # more records alive at once than the library's first P-copy pool holds (1024): the pool grew, keeping them
        assert peak > 1024, peak
        _sequences[name, n_cats] = trace
    return _sequences[name, n_cats]


@pytest.mark.gpu
@pytest.mark.parametrize("name,n_cats", LINEAGE)
def test_snapshot_lineage(name, n_cats, gpu_backend, monkeypatch):
    _lineage(name, n_cats, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("n_cats", [4, 1])
def test_lineage_same_bits_on_every_tiled_configuration(n_cats, gpu_backend, monkeypatch):
    """Same seed: tiled configurations with the same tiles per warp compute the same lnL sequence bit for bit (stack
    slots, spills, store path and records change no arithmetic); one tile per warp instead of two changes the order in
    which a thread's sites enter the block sum, so it and the row-major kernel agree to summation order."""
    seqs = {name: np.array(_lineage(name, c, monkeypatch)) for name, c in LINEAGE if c == n_cats}
    row, tiled = seqs.pop("row"), seqs.pop("tiled")
    for name, s in seqs.items():
        if LINEAGE_ENV[name].get("CYBAYES_S2T_V", "2") == "2":
            assert np.array_equal(s, tiled), name
        assert np.all(np.abs(s - row) <= 1e-13 * np.abs(row)), name
    assert np.all(np.abs(tiled - row) <= 1e-13 * np.abs(row))


@pytest.mark.gpu
def test_snapshot_lineage_at_the_tiled_threshold(gpu_backend, monkeypatch):
    """Unforced: 64 taxa x 81 920 patterns selects the tiled kernel by size (as test_cache_that_does_not_fit)."""
    _set_env(monkeypatch, {})
    trace, _ = run_lineage(_engine, 64, 81920, 4, 40, 33, reservoir=4, check_every=20, pull_every=8)
    assert len(trace) > 1 + 40


# ------------------------------------------------------------------------------------------------ weighted parity
def _weighted_engine(codes, S, C, amb, w, tree, tm):
    from cybayes_b200.engine import Engine
    eng = Engine(codes, S, C, amb, weights=w)
    ekeys = list(tree)
    block = eng.alloc_slots(len(ekeys) * C)
    slot_of = {(k, e): block.base + k * len(ekeys) + i for k in range(C) for i, e in enumerate(ekeys)}
    eng.upload_pmats(np.arange(block.base, block.base + block.n, dtype=np.int32),
                     np.stack([tm[k][e] for k in range(C) for e in ekeys]))
    return eng, slot_of


def _check_weighted(S, n_taxa, n_sites, model, n_cats=4, uint16=False):
    """lnL of a full pass (cache kept and likelihood only) and of a dirty path whose tip edge takes another edge's
    matrices, with random integer weights, against the weighted scaled oracle."""
    from cybayes_b200.likelihood import _Plan
    tree, root, edges, codes, amb, pi, er, rates = _random_problem(2000 + S, n_taxa, n_sites, S, n_cats=n_cats)
    if uint16:
        codes = codes.astype(np.uint16)
    w = _weights(np.random.default_rng(S * 7 + n_sites), n_sites)
    C = len(rates)
    tm = [oracle.prob_t(model, S == 2, pi, tree, er, r) for r in rates]
    leaves = _oracle_leaves(codes, S, amb)
    want = oracle.mat_ml_scaled(pi, root, leaves, edges, tm, n_sites, n_taxa, n_cats=C, weights=w)
    unweighted = oracle.mat_ml_scaled(pi, root, leaves, edges, tm, n_sites, n_taxa, n_cats=C)
    assert abs(want - unweighted) > 1e-6 * abs(want)
    eng, slot_of = _weighted_engine(codes, S, C, amb, w, tree, tm)
    plan = _Plan(edges)
    pslots = np.array([[slot_of[k, e] for k in range(C)] for e in plan.edge_keys], dtype=np.int32)
    lnl, snap = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=True, force_walk=True)
    info = eng.last_eval_info()
    assert abs(lnl - want) <= 1e-12 * abs(want), (lnl, want)
    only, _ = eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=False)
    assert only == lnl
    parents = oracle.parent_of(tree)
    ekeys = list(tree)
    for tip in (1, n_taxa):
        path = sorted(oracle.path_to_root(parents, tip, root), key=plan.index.__getitem__)
        other = ekeys[(tip * 7) % len(ekeys)]
        ch = np.array([c for n in path for c in plan.kids[n]], dtype=np.int32)
        ps = np.array([[slot_of[k, other if c == tip else (n, c)] for k in range(C)] for n in path for c in plan.kids[n]],
                      dtype=np.int32)
        got, _ = eng.eval(snap, np.array(path, dtype=np.int32), ch, ps, pi, want_snapshot=False)
        tm2 = [dict(t) for t in tm]
        for k in range(C):
            tm2[k][parents[tip], tip] = tm[k][other]
        want2 = oracle.mat_ml_scaled(pi, root, leaves, edges, tm2, n_sites, n_taxa, n_cats=C, weights=w)
        assert abs(got - want2) <= 1e-12 * abs(want2), (tip, got, want2)
    eng.release_snapshot(snap)
    eng.close()
    return info


WEIGHTED = [  # kernel family, S, taxa, patterns, model, n_cats, environment
    ("prune_s2_kernel", 2, 60, 1237, "F81", 4, {"CYBAYES_S2_TILED": "0"}),
    ("prune_s2_kernel", 2, 33, 700, "F81", 1, {"CYBAYES_S2_TILED": "0"}),
    ("prune_s2t_kernel_v1", 2, 60, 1237, "F81", 4, {"CYBAYES_S2_TILED": "1", "CYBAYES_S2T_V": "1"}),
    ("prune_s2t_kernel_v2", 2, 60, 1237, "F81", 4, {"CYBAYES_S2_TILED": "1", "CYBAYES_S2T_V": "2"}),
    ("prune_s2t_kernel_v2", 2, 90, 2101, "F81", 1, {"CYBAYES_S2_TILED": "1", "CYBAYES_S2T_V": "2"}),
    ("prune_general_kernel", 5, 12, 333, "GTR", 4, {}),
    ("prune_general_kernel_u16", 130, 6, 129, "F81", 4, {}),
    ("prune_dmma_kernel", 40, 9, 300, "GTR", 4, {"CYBAYES_DMMA_RC": "0"}),
    ("prune_dmma_rc_kernel", 64, 9, 200, "GTR", 4, {"CYBAYES_DMMA_RC": "1"}),
    ("prune_dmma_rc_kernel", 16, 9, 300, "GTR", 4, {"CYBAYES_DMMA_RC": "1"}),
]


@pytest.mark.gpu
@pytest.mark.parametrize("family,S,n_taxa,n_sites,model,n_cats,env", WEIGHTED)
def test_weighted_patterns_vs_oracle(family, S, n_taxa, n_sites, model, n_cats, env, gpu_backend, monkeypatch):
    _set_env(monkeypatch, env)
    info = _check_weighted(S, n_taxa, n_sites, model, n_cats=n_cats, uint16=family.endswith("_u16"))
    if family.startswith("prune_s2"):   # only the tiled kernel keeps small subtrees as records
        assert (info["small_records"] > 0) == family.startswith("prune_s2t")


@pytest.mark.gpu
@pytest.mark.parametrize("v", ["1", "2"])
def test_tiled_compressed_patterns_equal_the_alignment(v, gpu_backend, monkeypatch):
    """Tiled kernel: unique columns with their multiplicities (alignment.compress_patterns) against every column."""
    from cybayes_b200.alignment import compress_patterns
    _set_env(monkeypatch, {"CYBAYES_S2_TILED": "1", "CYBAYES_S2T_V": v})
    from cybayes_b200.likelihood import _Plan
    tree, root, edges, base, amb, pi, er, rates = _random_problem(77, 48, 900, 2)
    rng = np.random.default_rng(5)
    codes = np.ascontiguousarray(base[:, rng.integers(0, base.shape[1], size=6000)])
    pc, wc, smap = compress_patterns(codes)
    assert pc.shape[1] < 1000 and wc.max() > 3 and np.array_equal(pc[:, smap], codes)
    C = len(rates)
    tm = [oracle.prob_t("F81", True, pi, tree, er, r) for r in rates]
    plan = _Plan(edges)
    want = oracle.mat_ml_scaled(pi, root, _oracle_leaves(codes, 2, amb), edges, tm, codes.shape[1], 48, n_cats=C)
    got = []
    for cd, w in ((pc, wc), (codes, None)):
        eng, slot_of = _weighted_engine(cd, 2, C, amb, w, tree, tm)
        pslots = np.array([[slot_of[k, e] for k in range(C)] for e in plan.edge_keys], dtype=np.int32)
        got.append(eng.eval(None, plan.nodes, plan.children, pslots, pi, want_snapshot=False)[0])
        eng.close()
    assert abs(got[0] - got[1]) <= 1e-12 * abs(got[1]), got
    assert abs(got[0] - want) <= 1e-12 * abs(want), (got, want)


# ------------------------------------------------------------------------------------- recorded traces, tiled kernel
BINARY_TRACES = [t for t in TRACES if t[0] in ("binary_F81", "twoStates_F81", "twoStates_JC", "narrow_F81", "narrow_JC",
                                              "broad_F81")]


def _assert_tiled_engine():
    """The chain's engine runs the tiled kernel: a caterpillar's ((1, 2), 3) subtree is kept as a small-subtree record,
    which the row-major kernel never makes."""
    from cybayes_b200 import config, likelihood
    eng, _ = likelihood.engine_for(config.LEAF_LLMAT, config.N_CATS)
    N, C, S = eng.n_taxa, eng.n_cats, eng.n_states
    assert N >= 4 and S == 2
    nodes = np.arange(N + 1, 2 * N, dtype=np.int32)
    children = np.array([1, 2] + [x for i in range(3, N + 1) for x in (N + i - 2, i)], dtype=np.int32)
    block = eng.alloc_slots(C)
    slots = np.arange(block.base, block.base + C, dtype=np.int32)
    eng.upload_pmats(slots, np.stack([[[0.9, 0.1], [0.2, 0.8]]] * C))
    _, snap = eng.eval(None, nodes, children, np.tile(slots, (2 * (N - 1), 1)), np.array([0.4, 0.6]),
                       want_snapshot=True, force_walk=True)
    info = eng.last_eval_info()
    eng.release_snapshot(snap)
    assert info["small_records"] > 0, info


@pytest.mark.gpu
@pytest.mark.parametrize("runner", ["driver", "native"])
@pytest.mark.parametrize("name,n_gen", BINARY_TRACES)
def test_binary_trace_on_the_tiled_kernel(name, n_gen, runner, golden_cases, gpu_backend, tmp_path, monkeypatch):
    """The recorded reference traces (compare_trace, check_outputs) with the tiled 2-state kernel forced on."""
    _set_env(monkeypatch, {"CYBAYES_S2_TILED": "1"})
    (_driver_trace if runner == "driver" else _native_trace)(name, n_gen, golden_cases, gpu_backend, tmp_path)
    _assert_tiled_engine()


@pytest.mark.gpu
def test_likelihood_first_trace_on_the_tiled_kernel(golden_cases, gpu_backend, tmp_path, monkeypatch):
    """narrow_F81, native runner, likelihood-first full-table proposals (repeated with the cache on acceptance)."""
    _set_env(monkeypatch, {"CYBAYES_S2_TILED": "1", "CYBAYES_CHAIN_LNL_FIRST": "1"})
    _native_trace("narrow_F81", 3000, golden_cases, gpu_backend, tmp_path)
    _assert_tiled_engine()


@pytest.mark.gpu
def test_c1_at_its_stated_length_on_the_tiled_kernel(golden_cases, gpu_backend, tmp_path, monkeypatch):
    """Config C1's 100 000 recorded generations, native runner, tiled kernel forced on."""
    _set_env(monkeypatch, {"CYBAYES_S2_TILED": "1"})
    _c1_at_its_stated_length("native", golden_cases, gpu_backend, tmp_path)
    _assert_tiled_engine()
