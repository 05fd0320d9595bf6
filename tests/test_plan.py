"""The evaluation planner (cybayes_b200/csrc/plan.cpp) on the CPU: plans of seeded random trees, dirty paths and NNI /
SPR lists against snapshots, checked op by op against the rules the kernels rely on; the C4 plan's counters; and the
messages malformed lists fail with.  The planner is compiled with tests/plan_probe.cpp into a temporary directory."""
import importlib.util
import os
import subprocess
import sys
import sysconfig

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(REPO, "cybayes_b200", "csrc")
if REPO not in sys.path:
    sys.path.insert(0, REPO)

TIP, BUFFER, CARRIED, CHERRY, STACK, SMALL = range(6)
WANT_SNAPSHOT, STORE_ROOT, FORCE_LEVELS, FORCE_WALK, NO_FOLD = 1, 2, 8, 16, 32
# op columns of plan_probe.build
NODE, K0, R0, E0, K1, R1, E1, OUT_BUF, PF_BUF, IS_ROOT, KEEP, STREAM, SPILL, PUSHED, MAKE_REC, SYNTH = range(16)


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    pytest.importorskip("pybind11", reason="the planner probe is a pybind11 module")
    out = tmp_path_factory.mktemp("plan_probe")
    so = str(out / ("plan_probe" + sysconfig.get_config_var("EXT_SUFFIX")))
    inc = subprocess.run([sys.executable, "-m", "pybind11", "--includes"], check=True, capture_output=True,
                         text=True).stdout.split()
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wall", *inc, "-I", CSRC,
                    os.path.join(REPO, "tests", "plan_probe.cpp"), os.path.join(CSRC, "plan.cpp"), "-o", so], check=True)
    spec = importlib.util.spec_from_file_location("plan_probe", so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


# ---- configurations (one B200: 148 SMs)
def _cfg(**kw):
    c = dict(n_taxa=0, n_cats=4, code_bytes=1, P=81920, sm_count=148, family_s2=True, dmma_rc=False, s2_tiled=False,
             s2t_slots=0, s2t_bulk=False, s2t_prefetch=True, s2t_small_recs=True, stream_stores=True, tile_sites=256,
             tile_blocks=1, blocks_per_sm=3)
    states = kw.pop("n_states", 2)
    c.update(kw)
    c["buffer_bytes"] = c["n_cats"] * states * c["P"] * 8 + (1 if c["family_s2"] else c["n_cats"]) * c["P"] * 4
    return c


TILED = dict(s2_tiled=True, s2t_slots=3, tile_sites=256, blocks_per_sm=3)
CONFIGS = {
    "rowmajor": _cfg(P=40000),
    "rowmajor_small": _cfg(P=8192, blocks_per_sm=3),
    "tiled": _cfg(**TILED),
    "tiled_v1_minb4_1slot": _cfg(**{**TILED, "s2t_slots": 1, "blocks_per_sm": 4}),
    "tiled_bulk": _cfg(**TILED, s2t_bulk=True),
    "tiled_no_small_recs": _cfg(**TILED, s2t_small_recs=False),
    "tiled_c1_no_prefetch": _cfg(**TILED, n_cats=1, s2t_prefetch=False),
    "general": _cfg(family_s2=False, n_states=20, P=50048, tile_sites=32, tile_blocks=4, blocks_per_sm=2),
    "register_carried": _cfg(family_s2=False, n_states=24, P=2048, dmma_rc=True, tile_sites=128, tile_blocks=4,
                             blocks_per_sm=1),
}


# ---- trees: tips 1..N, internal nodes N+1..2N-1; kids[node] = [a, b], parent[node]
class Tree:
    def __init__(self, n, rng):
        self.n = n
        self.kids = {}
        self.parent = {}
        pool = list(range(1, n + 1))
        ids = list(rng.permutation(np.arange(n + 1, 2 * n)))
        while len(pool) > 1:
            i, j = rng.choice(len(pool), 2, replace=False)
            a, b = pool[i], pool[j]
            nd = int(ids.pop())
            self.kids[nd] = [a, b]
            self.parent[a] = self.parent[b] = nd
            pool = [x for k, x in enumerate(pool) if k not in (i, j)] + [nd]
        self.root = pool[0]
        self.parent[self.root] = 0

    def copy(self):
        t = Tree.__new__(Tree)
        t.n, t.root = self.n, self.root
        t.kids = {k: list(v) for k, v in self.kids.items()}
        t.parent = dict(self.parent)
        return t

    def postorder(self):
        out, stack = [], [(self.root, False)]
        while stack:
            nd, done = stack.pop()
            if nd <= self.n:
                continue
            if done:
                out.append(nd)
            else:
                stack += [(nd, True), (self.kids[nd][1], False), (self.kids[nd][0], False)]
        return out

    def ancestors(self, nd):
        out = []
        while nd:
            if nd > self.n:
                out.append(nd)
            nd = self.parent[nd]
        return out

    def _sub(self, nd):
        stack = [nd]
        while stack:
            x = stack.pop()
            yield x
            if x > self.n:
                stack += self.kids[x]

    def nni(self, rng):
        """Swap a child of internal non-root node v with v's sibling; returns v."""
        cand = [v for v in self.kids if v != self.root]
        v = int(rng.choice(cand))
        u = self.parent[v]
        si = 1 - self.kids[u].index(v)
        ci = int(rng.integers(2))
        s, c = self.kids[u][si], self.kids[v][ci]
        self.kids[u][si], self.kids[v][ci] = c, s
        self.parent[c], self.parent[s] = u, v
        return [v]

    def spr(self, rng):
        """Prune the subtree under x (with its parent p) and regraft it on another edge; returns the touched nodes."""
        cand = [x for x in self.parent if x != self.root and self.parent[x] != self.root]
        x = int(rng.choice(cand))
        p = self.parent[x]
        g = self.parent[p]
        s = self.kids[p][1 - self.kids[p].index(x)]
        sub = set(self._sub(p))
        targets = [b for b in self.parent if b not in sub and b != self.root and b != s]
        if not targets:
            return self.nni(rng)
        self.kids[g][self.kids[g].index(p)] = s
        self.parent[s] = g
        b = int(rng.choice(targets))
        a = self.parent[b]
        self.kids[a][self.kids[a].index(b)] = p
        self.parent[p] = a
        self.kids[p] = [x, b]
        self.parent[b] = p
        return [g, p]


def op_list(tree, nodes, rng):
    """(nodes, children) of the ops recomputing `nodes` (children before parents), children in random order."""
    ch = []
    for nd in nodes:
        a, b = tree.kids[nd]
        ch += [a, b] if rng.integers(2) else [b, a]
    return np.array(nodes, dtype=np.int32), np.array(ch, dtype=np.int32)


def dirty_nodes(tree, starts):
    on = set()
    for s in starts:
        on.update(tree.ancestors(s))
    return [nd for nd in tree.postorder() if nd in on]


# ---- snapshots: what eval_impl keeps of a plan
class Snap:
    def __init__(self, n_nodes, prev=None):
        self.buf = prev.buf.copy() if prev else np.full(n_nodes, -1, np.int32)
        self.rec = prev.rec.copy() if prev else np.full(n_nodes, -1, np.int32)

    def arrays(self):
        return (self.buf, self.rec)


def snapshot_after(plan, nodes, children, recs, prev, n_nodes):
    """The snapshot a cache-kept evaluation returns: kept partials, folded cherries and small-subtree records."""
    sn = Snap(n_nodes, prev)
    for op in plan["ops"]:
        if op[KEEP]:
            sn.buf[op[NODE]], sn.rec[op[NODE]] = 7, -1
        for k, r in ((K0, R0), (K1, R1)):
            if op[k] == CHERRY and op[r] >= 0:
                fo = op[r]
                recs.append((children[2 * fo], children[2 * fo + 1]))
                sn.buf[nodes[fo]], sn.rec[nodes[fo]] = -1, len(recs) - 1
        if op[MAKE_REC]:
            ids = [op[r] if op[k] == TIP else (nodes[op[r]] if op[r] >= 0 else ~op[r]) for k, r in ((K0, R0), (K1, R1))]
            recs.append(tuple(ids))
            sn.buf[op[NODE]], sn.rec[op[NODE]] = -1, len(recs) - 1
    return sn


def run(probe, cfg, lists, flags, snap=None, recs=(), split_env=0):
    offsets = np.cumsum([0] + [len(n) for n, _ in lists]).astype(np.int32)
    nodes = np.concatenate([n for n, _ in lists]).astype(np.int32)
    children = np.concatenate([c for _, c in lists]).astype(np.int32)
    r = np.array(recs, dtype=np.int32).reshape(-1, 2)
    plan = probe.build(cfg, None if snap is None else snap.arrays(), r, offsets, nodes, children, flags, split_env)
    return plan, offsets, nodes, children


# ---- the invariants
def check_plan(probe, cfg, plan, offsets, nodes, children, flags, snap, recs):
    assert "error" not in plan, plan.get("error")
    N, C = cfg["n_taxa"], cfg["n_cats"]
    ops, ranges, launches = plan["ops"], plan["ranges"], plan["launches"]
    n_lists = len(offsets) - 1
    total = offsets[-1]
    K = cfg["s2t_slots"] if cfg["s2_tiled"] else 0
    slot_base = probe.S2T_STAGING if cfg["s2t_bulk"] else 0
    tip_row = cfg["P"] * cfg["code_bytes"]

    def child_node(op, kx):   # node id of child kx from the caller's arrays or the record the op recomputes
        e = op[E0 if kx == 0 else E1]
        if e >= 0:
            return children[e]
        rec, k = divmod(~e, 2 * C)
        return recs[rec][k // C]

    # ranges and launches
    range_of = np.full(len(ops), -1)
    for ri, (b, e, out, _) in enumerate(ranges):
        assert b < e and (range_of[b:e] == -1).all()
        range_of[b:e] = ri
    launch_of_range = np.full(len(ranges), -1)
    for li_, (rb, re_, max_ops, n_bufs) in enumerate(launches):
        assert (launch_of_range[rb:re_] == -1).all()
        launch_of_range[rb:re_] = li_
        assert max_ops >= max(ranges[rb:re_, 1] - ranges[rb:re_, 0])
    assert (launch_of_range >= 0).all()

    # every caller op is exactly one of: a plan op, a folded cherry
    seen = np.zeros(total, int)
    for op in ops:
        if not op[SYNTH]:
            caller = op[E0] // 2
            assert op[E1] // 2 == caller and op[NODE] == nodes[caller]
            seen[caller] += 1
    folded = [op[r] for op in ops for k, r in ((K0, R0), (K1, R1)) if op[k] == CHERRY and op[r] >= 0]
    seen[folded] += 1
    assert (seen == 1).all() and len(set(folded)) == len(folded) == plan["n_cherries"]
    if flags & NO_FOLD or not cfg["family_s2"]:
        assert plan["n_cherries"] == 0

    # the root of each list is last in its range and carries the list's out_index
    for li in range(n_lists):
        rr = [ri for ri in range(len(ranges)) if ranges[ri, 2] == li]
        assert len(rr) == 1
        root = ops[ranges[rr[0], 1] - 1]
        assert root[IS_ROOT] and root[NODE] == nodes[offsets[li + 1] - 1]
    assert ops[:, IS_ROOT].sum() == n_lists

    launch = lambda p: launch_of_range[range_of[p]]  # noqa: E731
    n_tip = n_cherry = n_reads = n_stack = n_small = 0
    stacks = {}
    for p, op in enumerate(ops):
        if range_of[p] < 0:   # not run: an inlined subtree's descriptor
            assert not op[KEEP] and not op[PUSHED] and op[OUT_BUF] < 0
        if cfg["s2_tiled"]:
            assert probe.s2t_rank(op[K0]) <= probe.s2t_rank(op[K1]) and probe.s2t_combo(op[K0], op[K1]) >= 0
        st = stacks.setdefault(range_of[p], [])
        for kx, (k, r) in enumerate(((K0, R0), (K1, R1))):
            kind, ref, ch = op[k], op[r], child_node(op, kx)
            if kind == TIP:
                assert ref == ch and 1 <= ch <= N
                n_tip += 1
            elif kind == CARRIED:
                assert range_of[p] >= 0 and p > ranges[range_of[p], 0] and ops[p - 1, NODE] == ch
            elif kind == STACK and not (kx == 1 and op[PF_BUF] >= 0):
                assert st and st[-1] == (ref, ch), "stack pops must match pushes, last in first out"
                st.pop()
                n_stack += 1
            elif kind in (BUFFER, STACK):   # a stored partial, read directly or through a prefetch buffer
                if kind == STACK:
                    assert op[K0] == CARRIED
                if ref < 0:
                    assert ~ref == ch and snap is not None and snap.buf[ch] >= 0
                else:
                    src = ops[ref]
                    assert src[NODE] == ch and src[KEEP] and range_of[ref] >= 0
                    if kind == STACK:
                        assert launch(ref) < launch(p) or range_of[ref] != range_of[p]
                    else:
                        assert launch(ref) < launch(p) or (range_of[ref] == range_of[p] and ref < p and src[SPILL])
                n_reads += 1
            elif kind == CHERRY:
                if ref >= 0:
                    assert nodes[ref] == ch
                else:
                    assert ~ref == ch and snap is not None and snap.rec[ch] >= 0
                n_cherry += 1
            elif kind == SMALL:
                assert cfg["s2_tiled"] and ops[ref, NODE] == ch and range_of[ref] < 0 and not ops[ref, KEEP]
                n_small += 1
            else:
                raise AssertionError(f"bad child kind {kind}")
        if op[PUSHED]:
            assert range_of[p] >= 0 and slot_base <= op[OUT_BUF] < slot_base + K
            st.append((op[OUT_BUF], op[NODE]))
    assert all(not s for s in stacks.values()), "every push is popped in its range"

    # a range's order needs the fewest read-backs possible with K stack slots: per op, visit one child first and push it
    # (or read it back when no slot is free) and carry the other, or read the first back to leave the second every slot
    for b, e, _, _ in ranges:
        f = {}
        spills = 0
        for p in range(b, e):
            kids = []
            for k, r in ((K0, R0), (K1, R1)):
                kind, ref = ops[p, k], ops[p, r]
                if kind == CARRIED:
                    kids.append(p - 1)
                elif kind == STACK and not (k == K1 and ops[p, PF_BUF] >= 0):
                    kids.append(next(q for q in range(p - 1, b - 1, -1) if ops[q, PUSHED] and ops[q, OUT_BUF] == ref
                                     and ops[q, NODE] == child_node(ops[p], 0 if k == K0 else 1)))
                elif kind == BUFFER and ref >= 0 and range_of[ref] == range_of[p]:
                    kids.append(ref)
                    spills += 1
            if len(kids) == 2:
                fa, fb = f[kids[0]], f[kids[1]]
                f[p] = [min(fa[k] + (k == 0) + fb[max(k - 1, 0)], fb[k] + (k == 0) + fa[max(k - 1, 0)],
                            fa[k] + 1 + fb[k] if k > 0 else 1 << 30) for k in range(K + 1)]
            else:
                f[p] = f[kids[0]] if kids else [0] * (K + 1)
        assert spills == f[e - 1][K], "read-backs inside a range are not the fewest possible"

    # counters
    assert plan["n_stored"] == ops[:, KEEP].sum()
    assert plan["n_spills"] == (ops[:, KEEP] & ops[:, SPILL]).sum()
    assert plan["n_small_recs"] == ops[:, MAKE_REC].sum()
    assert plan["n_stack"] == n_stack and plan["n_buffer_reads"] == n_reads and plan["n_inlined"] == n_small
    assert plan["bytes_written"] == plan["n_stored"] * cfg["buffer_bytes"]
    assert plan["bytes_read"] == (n_tip + 2 * n_cherry) * tip_row + n_reads * cfg["buffer_bytes"] + n_lists * cfg["P"] * 8
    if not flags & WANT_SNAPSHOT:
        assert not ops[:, MAKE_REC].any()

    # each launch's n_bufs covers every tile buffer its ops name
    for rb, re_, _, n_bufs in launches:
        for b, e, _, _ in ranges[rb:re_]:
            for op in ops[b:e]:
                assert op[OUT_BUF] < n_bufs and op[PF_BUF] < n_bufs
                for k, r in ((K0, R0), (K1, R1)):
                    if op[k] == STACK and op[PF_BUF] < 0:
                        assert op[r] < n_bufs


CASES = [(name, flags, split) for name in CONFIGS
         for flags, split in ((WANT_SNAPSHOT, 0), (0, 0), (WANT_SNAPSHOT | STORE_ROOT, 0), (WANT_SNAPSHOT | FORCE_LEVELS, 0),
                              (WANT_SNAPSHOT | FORCE_WALK, 0), (WANT_SNAPSHOT, 9))]


@pytest.mark.parametrize("name,flags,split_env", CASES)
def test_plan_invariants(probe, name, flags, split_env):
    """Full passes, then dirty paths, NNI and SPR lists and batches against the snapshots the passes leave."""
    rng = np.random.default_rng([sum(map(ord, name)), flags, split_env])
    for n_taxa in (5, 17, 64, 150, 300):
        cfg = dict(CONFIGS[name], n_taxa=n_taxa)
        tree = Tree(n_taxa, rng)
        nodes, children = op_list(tree, tree.postorder(), rng)
        recs = []
        for f in (flags, flags & ~WANT_SNAPSHOT):
            plan, off, nv, cv = run(probe, cfg, [(nodes, children)], f, split_env=split_env)
            check_plan(probe, cfg, plan, off, nv, cv, f, None, recs)
        plan, off, nv, cv = run(probe, cfg, [(nodes, children)], flags | WANT_SNAPSHOT, split_env=split_env)
        snap = snapshot_after(plan, nv, cv, recs, None, 2 * n_taxa)
        for step in range(12):
            t2 = tree.copy()
            move = step % 3
            starts = ([int(x) for x in rng.integers(1, 2 * n_taxa, rng.integers(1, 4))] if move == 0
                      else t2.nni(rng) if move == 1 else t2.spr(rng))
            nd2, ch2 = op_list(t2, dirty_nodes(t2, starts), rng)
            f = (flags & (FORCE_LEVELS | FORCE_WALK)) | (WANT_SNAPSHOT if step % 2 else 0) | (STORE_ROOT if step % 4 == 1 else 0)
            plan, off, nv, cv = run(probe, cfg, [(nd2, ch2)], f, snap, recs, split_env)
            check_plan(probe, cfg, plan, off, nv, cv, f, snap, recs)
            if f & WANT_SNAPSHOT:   # accept: the next lists run against the new snapshot and tree
                snap = snapshot_after(plan, nv, cv, recs, snap, 2 * n_taxa)
                tree = t2
            if not flags & FORCE_LEVELS:   # a batch of candidates (cb_eval_batch: no flags)
                batch = []
                for _ in range(3):
                    t3 = tree.copy()
                    st3 = t3.nni(rng) if rng.integers(2) else [int(rng.integers(1, 2 * n_taxa))]
                    if dirty_nodes(t3, st3):
                        batch.append(op_list(t3, dirty_nodes(t3, st3), rng))
                plan, off, nv, cv = run(probe, cfg, batch, 0, snap, recs, split_env)
                check_plan(probe, cfg, plan, off, nv, cv, 0, snap, recs)


def test_c4_plan_counters(probe):
    """bench.py's C4 full step planned for one B200 gives the counters the B200 measured
    (profiles/r03_bench_c4_ab_branch.jsonl)."""
    from cybayes_b200.likelihood import _plan_for
    from cybayes_b200.synthetic import SyntheticAlignment
    edges = SyntheticAlignment(1024, 1_000_000, 2, 20260101, block_sites=125000).edge_order()
    p = _plan_for(edges)
    cfg = _cfg(n_taxa=1024, P=1_000_000, **TILED)
    plan, off, nv, cv = run(probe, cfg, [(np.asarray(p.nodes), np.asarray(p.children))], WANT_SNAPSHOT)
    check_plan(probe, cfg, plan, off, nv, cv, WANT_SNAPSHOT, None, [])
    counts = dict(ops=len(plan["ops"]) - plan["n_inlined"], stored=plan["n_stored"], read_back=plan["n_buffer_reads"],
                  stack_pops=plan["n_stack"], spills=plan["n_spills"], cherries_folded=plan["n_cherries"],
                  small_records=plan["n_small_recs"], launches=len(plan["launches"]))
    assert counts == dict(ops=544, stored=460, read_back=5, stack_pops=143, spills=0, cherries_folded=351,
                          small_records=211, launches=2)


def _caterpillar(n):
    """Op list of ((1, 2), 3), 4) ...: nodes n+1 .. 2n-1."""
    nodes = np.arange(n + 1, 2 * n, dtype=np.int32)
    ch = [1, 2] + [x for i in range(1, n - 1) for x in (n + i, i + 2)]
    return nodes, np.array(ch, dtype=np.int32)


def test_plan_errors(probe):
    cfg = dict(CONFIGS["tiled"], n_taxa=8)
    nodes, ch = _caterpillar(8)

    def err(lists, flags=0, snap=None):
        plan, *_ = run(probe, cfg, lists, flags, snap)
        return plan.get("error")

    bad = ch.copy()
    bad[3] = 16
    assert err([(nodes, bad)]) == "op 1: bad child id 16"
    bad[3] = 0
    assert err([(nodes, bad)]) == "op 1: bad child id 0"
    assert err([(np.r_[nodes[:3], nodes[2:]], np.r_[ch[:6], ch[4:]])]) == "op 3: node 11 is computed twice"
    swapped_n, swapped_c = nodes.copy(), ch.copy()
    swapped_n[[1, 2]] = swapped_n[[2, 1]]
    swapped_c[[2, 3, 4, 5]] = swapped_c[[4, 5, 2, 3]]
    assert err([(swapped_n, swapped_c)]) == "op 1: child 10 is computed after its parent"
    assert err([(nodes[3:], ch[6:])]) == "op 0: child 11 is neither recomputed nor in the input snapshot"
    # batch candidates: a chain is required under forced levels, and every op must lie under the candidate's root
    tree = Tree(8, np.random.default_rng(1))
    full = op_list(tree, tree.postorder(), np.random.default_rng(2))
    assert err([full, full], FORCE_LEVELS) == "cb_eval_batch: candidate 0 is not a chain (level schedule forced)"
    snap = Snap(16)
    snap.buf[9:16] = 1
    two = (np.array([9, 10], np.int32), np.array([1, 2, 3, 4], np.int32))
    assert err([(nodes[:1], ch[:2]), two], 0, snap) == "cb_eval_batch: candidate 1 has ops that are not under its root"
