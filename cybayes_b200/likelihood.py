"""Tree log-likelihood surfaces: ``matML`` / ``cache_matML`` of ML_gamma.pyx and ML.pyx on the GPU.

The reference walks the edge list in Python and calls NumPy ``dot`` per edge and category
(ML_gamma.pyx:22-38).  Here the edge list is turned once into a node-operation list
(children before parents), the P-matrix slots of every (edge, category) are gathered, and one
``cb_eval`` call runs the whole pass on the device: one launch per tree level for a full
evaluation, a single launch for a dirty path.  The returned cache is an opaque device
snapshot (the driver only hands it back, mat_mcmc_gamma.py:52,149,196); indexing it
(``cache[k][node]``) downloads the reference-shaped (S, n_sites) array.
"""
from __future__ import annotations

import os
from operator import itemgetter

import numpy as np

from . import config, subst
from .alignment import LeafMatrices, compress_patterns, compress_patterns_gpu
from .engine import Engine
from .subst import PMatTable

# ---------------------------------------------------------------------------- engines
_engines = {}  # (id(ll_mats), n_cats) -> (ll_mats, Engine, site_to_pattern or None)
# Pattern compression: alignments of up to COMPRESS_MAX_SITES columns are compressed on the host; longer ones on the GPU
# unless CYBAYES_COMPRESS_GPU=0.  COMPRESS_MAX_SITES = 0 switches compression off (every column is evaluated, weights 1).
COMPRESS_MAX_SITES = int(os.environ.get("CYBAYES_COMPRESS_MAX_SITES", "250000"))
COMPRESS_GPU = os.environ.get("CYBAYES_COMPRESS_GPU", "1") != "0"
_engine_factory = Engine  # tests substitute a fake engine here


def _codes_from_dense(ll_mats, n_taxa):
    """State codes from reference-style 0/1 float matrices (any dict id -> (S, P) array)."""
    first = np.asarray(ll_mats[1])
    S, P = first.shape
    amb_index, amb_rows = {}, [np.ones(S)]
    codes = np.empty((n_taxa, P), dtype=np.int64)
    weights_vec = np.arange(S)
    for t in range(1, n_taxa + 1):
        m = np.asarray(ll_mats[t])
        if m.shape != (S, P) or not np.isin(m, (0.0, 1.0)).all():
            raise ValueError("leaf matrices must be 0/1 arrays of shape (n_states, n_sites)")
        count = m.sum(axis=0)
        code = (m * weights_vec[:, None]).sum(axis=0).astype(np.int64)
        code[count == S] = S
        for p in np.nonzero((count != 1) & (count != S))[0]:
            members = tuple(np.nonzero(m[:, p])[0])
            if not members:
                raise ValueError("leaf column with no admissible state")
            if members not in amb_index:
                amb_index[members] = len(amb_rows)
                amb_rows.append(m[:, p].astype(np.float64))
            code[p] = S + amb_index[members]
        codes[t - 1] = code
    dtype = np.uint8 if S + len(amb_rows) <= 256 else np.uint16
    return codes.astype(dtype), S, np.array(amb_rows)


def engine_for(ll_mats, n_cats):
    """The device context holding `ll_mats` (uploaded once, keyed on object identity -- the
    driver always passes the same config.LEAF_LLMAT, mat_mcmc_gamma.py:55,149)."""
    key = (id(ll_mats), int(n_cats))
    hit = _engines.get(key)
    if hit is not None and hit[0] is ll_mats:
        return hit[1], hit[2]
    if isinstance(ll_mats, LeafMatrices):
        codes, S, amb = ll_mats.codes, ll_mats.n_states, ll_mats.amb_sets
    else:
        codes, S, amb = _codes_from_dense(ll_mats, len(ll_mats))
    site_map, weights = None, None
    if 0 < codes.shape[1] <= COMPRESS_MAX_SITES or (COMPRESS_MAX_SITES > 0 and COMPRESS_GPU):
        # short alignments: NumPy on the host; long ones (where np.unique over 1 KB columns takes minutes): column
        # hashing + verification on the GPU (same patterns, same order, same weights)
        if codes.shape[1] <= COMPRESS_MAX_SITES or _engine_factory is not Engine:
            pat, w, smap = compress_patterns(codes)
        else:
            pat, w, smap = compress_patterns_gpu(codes)
        if pat.shape[1] < codes.shape[1]:
            codes, weights, site_map = pat, w, smap
    rank, world = _shard_rank()
    if world > 1:
        # site-pattern sharding: this process (one per GPU) keeps a contiguous slice of the patterns; the
        # library all-reduces the scalar lnL over NCCL, so every rank sees the same number
        from .synthetic import shard_bounds
        cuts = [shard_bounds(codes.shape[1], r, world, 64) for r in range(world)]
        if any(h <= l for l, h in cuts):   # evaluated identically on every rank: all raise together, nobody is
            raise ValueError(              # left waiting inside the communicator set-up
                f"alignment has too few patterns ({codes.shape[1]}) to shard over {world} GPUs")
        lo, hi = cuts[rank]
        codes = np.ascontiguousarray(codes[:, lo:hi])
        weights = None if weights is None else np.ascontiguousarray(weights[lo:hi])
        site_map = None  # per-site read-back of partials is a single-GPU debugging aid
    eng = _engine_factory(codes, S, n_cats, amb, weights)
    if world > 1:
        global _comm_serial
        _comm_serial += 1
        uid, published = _nccl_id(eng, rank, f"{S}x{n_cats}x{_comm_serial}")
        eng.comm_init(uid, rank, world)     # collective: when it returns on rank 0 every rank has read the id
        if published is not None:
            try:
                os.remove(published)
            except OSError:
                pass
    _engines[key] = (ll_mats, eng, site_map)
    return eng, site_map


def _shard_rank():
    """(rank, world) when CYBAYES_SHARD=1 and the process was started by torchrun / mpirun-style env."""
    if os.environ.get("CYBAYES_SHARD", "0") != "1":
        return 0, 1
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def refuse_sharded_site_lnl():
    """Per-column log-likelihoods need every pattern and the column -> pattern map; a site-sharded rank has neither."""
    if os.environ.get("CYBAYES_SHARD", "0") == "1":
        raise ValueError("per-site log-likelihoods are not available with CYBAYES_SHARD=1: each rank holds only its "
                         "slice of the patterns (Engine.eval_sites returns that slice)")


_comm_serial = 0          # sharded contexts created by this process; never reset (reset_engines included)
_PROCESS_START = None


def _nccl_id(eng, rank, tag):
    """NCCL unique id made by rank 0 and handed to the other ranks through a file (no torch needed):
    CYBAYES_NCCL_ID_DIR (default: the system temp dir) / cybayes_nccl_<MASTER_PORT>_<launcher pid>_<tag>.id
    `tag` carries a per-process serial number, so two sharded alignments of one launch never share a name; readers
    ignore a file older than their own process (left behind by a dead launch with a recycled pid / port), rank 0
    removes such a file before it publishes and removes its own once every rank has joined (comm_init returns)."""
    import tempfile
    import time
    global _PROCESS_START
    if _PROCESS_START is None:
        try:
            import psutil
            _PROCESS_START = psutil.Process().create_time()
        except Exception:
            _PROCESS_START = time.time() - 3600.0
    d = os.environ.get("CYBAYES_NCCL_ID_DIR", tempfile.gettempdir())
    # all ranks of one launch share the parent (the torchrun agent): its pid keeps launches apart
    path = os.path.join(d, f"cybayes_nccl_{os.environ.get('MASTER_PORT', '0')}_{os.getppid()}_{tag}.id")
    if rank == 0:
        if os.path.exists(path):
            os.remove(path)
        uid = eng.nccl_unique_id()
        with open(path + ".tmp", "wb") as fh:
            fh.write(uid)
        os.replace(path + ".tmp", path)
        return uid, path
    t0 = time.time()
    while True:
        try:
            if os.path.getmtime(path) >= _PROCESS_START - 2.0:
                with open(path, "rb") as fh:
                    uid = fh.read()
                if len(uid) == 128:
                    return uid, None
        except OSError:
            pass
        if time.time() - t0 > 120:
            raise TimeoutError(f"rank 0 never published {path}")
        time.sleep(0.01)


def _default_engine(n_cats=None):
    """Engine of the driver's alignment (config.LEAF_LLMAT) for the substitution builders."""
    eng, _ = engine_for(config.LEAF_LLMAT, config.N_CATS if n_cats is None else n_cats)
    return eng


subst._engine_hook = _default_engine


def drop_engine(ll_mats):
    """Free the device contexts holding `ll_mats` (a driver that loads another alignment)."""
    for key in [k for k, v in _engines.items() if v[0] is ll_mats]:
        try:
            _engines.pop(key)[1].close()
        except Exception:
            pass


def reset_engines():
    """Drop every device context (tests, or a driver that loads another alignment)."""
    for _, eng, _ in _engines.values():
        try:
            eng.close()
        except Exception:
            pass
    _engines.clear()


# ------------------------------------------------------------------------------ plans
class _Plan:
    """Edge list -> node operations.  `nodes[i]` is completed by the i-th op in the order in
    which the reference finishes parents while walking `edges` (ML_gamma.pyx:24-36)."""
    __slots__ = ("edges", "node_list", "kids", "index", "_nodes", "_children", "_edge_keys", "_paths", "_perms")

    def __init__(self, edges):
        self.edges = list(edges)
        first, kids, node_list = {}, {}, []
        get = first.get
        for parent, child in self.edges:
            c0 = get(parent)
            if c0 is None:
                first[parent] = child
            else:
                kids[parent] = (c0, child)
                node_list.append(parent)
        if 2 * len(kids) != len(self.edges):
            raise ValueError("every internal node needs exactly two child edges")
        self.kids, self.node_list = kids, node_list
        self.index = dict(zip(node_list, range(len(node_list))))
        self._nodes = self._children = self._edge_keys = None
        self._paths = {}   # dirty set -> (nodes, children, edge keys, getter): the same few paths recur while a tree lives
        self._perms = []   # (key order of a transition-matrix table, positions of this plan's edges in it), MRU

    @property
    def nodes(self):
        if self._nodes is None:
            self._nodes = np.array(self.node_list, dtype=np.int32)
        return self._nodes

    @property
    def children(self):
        if self._children is None:
            kids = self.kids
            self._children = np.array([c for n in self.node_list for c in kids[n]], dtype=np.int32)
        return self._children

    @property
    def edge_keys(self):
        if self._edge_keys is None:
            kids = self.kids
            self._edge_keys = [(n, c) for n in self.node_list for c in kids[n]]
        return self._edge_keys


    def perm_for(self, src):
        """Positions of this plan's edges (op order) in `src`, the key order of a table that holds exactly these edges;
        None when it holds other edges.  A chain hands over tables in the same key order evaluation after evaluation
        (the order of its tree dict), so the match is one list comparison -- pointer-equal tuples mostly -- instead of
        one dict lookup per edge and category."""
        perms = self._perms
        for i, (keys, perm) in enumerate(perms):
            if keys is src or keys == src:
                if i:
                    perms.insert(0, perms.pop(i))
                return perm
        edge_keys = self.edge_keys
        if len(src) != len(edge_keys):
            return None
        where = dict(zip(src, range(len(src))))
        try:
            perm = np.fromiter(map(where.__getitem__, edge_keys), dtype=np.int32, count=len(edge_keys))
        except KeyError:
            return None
        perms.insert(0, (src, perm))
        del perms[4:]
        return perm


_plan_cache = []  # small MRU list of plans, matched by list equality


def _plan_for(edges):
    for i, p in enumerate(_plan_cache):
        if p.edges == edges:
            if i:
                _plan_cache.insert(0, _plan_cache.pop(i))
            return p
    p = _Plan(edges)
    _plan_cache.insert(0, p)
    del _plan_cache[4:]
    return p


try:   # optional CPython helper (csrc/hostgather.c): same bytes as the bytes.join route below, ~10x faster
    from . import _hostgather
except ImportError:   # not built: host-side glue only, the join route gives identical arrays
    _hostgather = None


def _gather_host_matrices(vals, n, S, out=None):
    """(n * S * S,) float64 array (`out` when given) from n reference-style (S, S) ndarrays.  The packed copy goes
    through _hostgather.pack (reads the array structs, ~10 ns per matrix) or, when that module is not built,
    bytes.join (buffer protocol, ~100 ns per matrix; np.concatenate needs ~320 ns); both refuse anything but
    contiguous float64 arrays, which then take the general route (other dtypes, views, nested lists)."""
    if out is None:
        out = np.empty(n * S * S, dtype=np.float64)
    if _hostgather is not None:
        if _hostgather.pack(vals, out):
            return out
    else:
        try:
            if vals[0].dtype == np.float64 and vals[-1].dtype == np.float64:
                buf = b"".join(vals)
                if len(buf) == n * S * S * 8:
                    out[:] = np.frombuffer(buf, dtype=np.float64)
                    return out
        except (AttributeError, TypeError, BufferError, ValueError):
            pass
    mats = np.array([np.asarray(v, dtype=np.float64) for v in vals])
    if mats.shape != (n, S, S):
        raise ValueError(f"transition matrices must be {S} x {S}")
    out[:] = mats.ravel()
    return out


def _slot_matrix(engine, tmats, edge_keys, getter=None, plan=None):
    """(n_edges, C) int32 P-slot table for the ops' edges.  Device tables are looked up; reference-style host dicts
    of ndarrays are gathered and uploaded with ONE host -> device copy for all categories.  With `plan` (full
    evaluations) a table that holds exactly the plan's edges is taken in its own key order and mapped onto the op
    order by the plan's cached permutation; anything else goes edge by edge through `getter`."""
    cols = []
    keep = []
    n = len(edge_keys)
    S = engine.n_states
    n_host = sum(1 for t in tmats if not isinstance(t, PMatTable))
    packed = None
    if n_host:
        # one packing buffer per engine, reused: upload_pmats has copied it into pinned staging when it returns, and a
        # fresh 134 MB array per call (C5) would cost 32 000 page faults before a single matrix is packed
        need = n_host * n * S * S
        buf = getattr(engine, "_pack_buf", None)
        if buf is None or buf.size < need:
            buf = engine._pack_buf = np.empty(need, dtype=np.float64)
        packed = buf[:need].reshape(n_host, n * S * S)
    host = []   # (column index, permutation or None) of the host-side categories, in the order of `packed`
    for t in tmats:
        if isinstance(t, PMatTable):
            if t.engine is not engine:
                raise ValueError("transition matrices belong to a different alignment")
            run = t.pristine() if plan is not None else None
            perm = plan.perm_for(run[0]) if run is not None else None
            if perm is not None:
                cols.append(perm + np.int32(run[1]))
                continue
            if getter is None:
                getter = itemgetter(*edge_keys) if n > 1 else (lambda d: (d[edge_keys[0]],))
            cols.append(getter(t._slots))
            continue
        out = packed[len(host)]
        perm = None
        if plan is not None and type(t) is dict and len(t) == n:
            if _hostgather is not None:    # a key order seen before: keys checked and values packed in one pass
                for keys, known in plan._perms:
                    if _hostgather.pack_dict(t, keys, out):
                        perm = known
                        break
            if perm is None:
                perm = plan.perm_for(list(t))
                if perm is not None:
                    _gather_host_matrices(list(t.values()), n, S, out)
        if perm is None:
            if getter is None:
                getter = itemgetter(*edge_keys) if n > 1 else (lambda d: (d[edge_keys[0]],))
            _gather_host_matrices(getter(t), n, S, out)
        host.append((len(cols), perm))
        cols.append(None)
    if host:
        block = engine.alloc_slots(n * n_host)
        keep.append(block)
        slots = np.arange(block.base, block.base + block.n, dtype=np.int32)
        engine.upload_pmats(slots, packed)
        for j, (col, perm) in enumerate(host):
            run = slots[j * n:(j + 1) * n]
            cols[col] = run if perm is None else run[perm]
    return np.ascontiguousarray(np.array(cols, dtype=np.int32).T), keep


class _CategoryView:
    def __init__(self, cache, k):
        self._cache, self._k = cache, k

    def __getitem__(self, node):
        return self._cache.partial(node)[self._k]

    def keys(self):
        return self._cache.nodes()


class PartialCache:
    """Opaque snapshot of all internal-node partials on the device (the second return value of
    matML / cache_matML).  ``cache[k][node]`` gives the reference's (S, n_sites) array.

    Deviations from the reference's list of dicts (ML_gamma.pyx:38-39), none visible to its drivers, which only
    hand the cache back: the ROOT partial is not stored unless CYBAYES_STORE_ROOT=1 (the fused root kernel does not
    need it; ``cache[k][root]`` raises otherwise); in site-sharded mode a rank only holds -- and returns -- its
    own slice of the patterns; and matML divides by the number of tables passed (len(tmats)), which is what the
    reference's drivers pass as n_cats."""

    def __init__(self, engine, snap, site_map, node_ids):
        self.engine, self.snap, self._site_map, self._nodes = engine, snap, site_map, node_ids

    def partial(self, node):
        a = self.engine.read_partial(self.snap, node)
        return a if self._site_map is None else a[:, :, self._site_map]

    def partial_scaled(self, node):
        a, e = self.engine.read_partial(self.snap, node, with_scale=True)
        if self._site_map is not None:
            a, e = a[:, :, self._site_map], e[self._site_map]
        return a, e

    def nodes(self):
        return list(self._nodes)

    def __getitem__(self, k):
        if not 0 <= k < self.engine.n_cats:
            raise IndexError(k)
        return _CategoryView(self, k)

    def __len__(self):
        return self.engine.n_cats

    def __del__(self):
        try:
            self.engine.release_snapshot(self.snap)
        except Exception:
            pass


STORE_ROOT = os.environ.get("CYBAYES_STORE_ROOT", "0") == "1"
# Speculative evaluation: on alignments with at least this many patterns a *full* pass first computes
# only lnL (no partial is written except the few the walk must read back); the cache is produced by a
# second, storing pass only if somebody uses it -- i.e. only if the proposal is accepted.  Most full-pass
# proposals (pi, rates, alpha, SPR) are rejected, so this trades one cheap pass for an expensive one.
LAZY_CACHE_MIN_SITES = int(os.environ.get("CYBAYES_LAZY_CACHE_MIN_SITES", str(1 << 62)))


CACHE_CHECK_MIN_BYTES = 1 << 30


def _cache_fits(engine, n_nodes):
    """Can this context hold one more full cache (one partial buffer per stored node) next to what it already has?
    Only asked when the cache is big enough to matter (> 1 GB); the margin covers temporaries of later dirty paths.
    C5 on one B200 (209 GB of partials) does not fit: matML then evaluates the likelihood without keeping partials
    and returns a LazyPartialCache that materialises on first use -- or fails there with a clear out-of-memory message."""
    mem = getattr(engine, "mem_info", None)
    if mem is None:
        return True
    info = mem()
    need = (n_nodes - 1) * info["partial"]
    if need < CACHE_CHECK_MIN_BYTES:
        return True
    return need <= 0.92 * (info["free"] + info["pooled"])


class LazyPartialCache(PartialCache):
    """Cache of a full pass whose partials are only materialised (by re-running the pass with
    stores) when first needed.  Holds what that needs: the op list, the P slots (kept alive through
    their owners) and pi as they were at evaluation time."""

    def __init__(self, engine, site_map, node_ids, plan, pslots, pi, keepalive):
        self.engine, self._site_map, self._nodes = engine, site_map, node_ids
        self._plan, self._pslots, self._pi, self._keep = plan, pslots, np.array(pi, dtype=np.float64), keepalive
        self._snap = None

    @property
    def snap(self):
        if self._snap is None:
            _, self._snap = self.engine.eval(None, self._plan.nodes, self._plan.children, self._pslots, self._pi,
                                             want_snapshot=True, store_root=STORE_ROOT)
            self._keep = None
        return self._snap

    def __del__(self):
        if self._snap is not None:
            try:
                self.engine.release_snapshot(self._snap)
            except Exception:
                pass


def _full(pi, root, ll_mats, edges, tmats, n_cats_tables):
    engine, site_map = engine_for(ll_mats, n_cats_tables)
    plan = _plan_for(edges)
    if plan.nodes[-1] != root:
        raise KeyError(root)
    pslots, keep = _slot_matrix(engine, tmats, plan.edge_keys, plan=plan)
    nodes = plan.nodes if STORE_ROOT else plan.nodes[:-1]
    if engine.n_patterns >= LAZY_CACHE_MIN_SITES or not _cache_fits(engine, len(plan.nodes)):
        lnl, _ = engine.eval(None, plan.nodes, plan.children, pslots, np.asarray(pi, dtype=np.float64),
                             want_snapshot=False)
        alive = keep + [t._block for t in tmats if isinstance(t, PMatTable)] + \
            [o for t in tmats if isinstance(t, PMatTable) for o in t._owners.values()]
        return np.float64(lnl), LazyPartialCache(engine, site_map, nodes.tolist(), plan, pslots, pi, alive)
    lnl, snap = engine.eval(None, plan.nodes, plan.children, pslots, np.asarray(pi, dtype=np.float64),
                            want_snapshot=True, store_root=STORE_ROOT)
    return np.float64(lnl), PartialCache(engine, snap, site_map, nodes.tolist())


def _dirty(pi, root, ll_mats, cache, nodes_recompute, edges, tmats, n_cats_tables):
    engine, site_map = engine_for(ll_mats, n_cats_tables)
    if not isinstance(cache, PartialCache) or cache.engine is not engine:
        raise TypeError("cache_LL_Mats must be the cache returned by matML/cache_matML for this alignment")
    plan = _plan_for(edges)
    key = (root,) + tuple(nodes_recompute)
    hit = plan._paths.get(key)
    if hit is None:
        index, kids = plan.index, plan.kids
        todo = sorted(set(nodes_recompute), key=index.__getitem__)
        if not todo or todo[-1] != root:
            todo = sorted(set(todo) | {root}, key=index.__getitem__)  # the root partial is never cached
        edge_keys = [(n, c) for n in todo for c in kids[n]]
        hit = plan._paths[key] = (np.array(todo, dtype=np.int32),
                                  np.array([c for n in todo for c in kids[n]], dtype=np.int32), edge_keys,
                                  itemgetter(*edge_keys) if len(edge_keys) > 1 else None)
        if len(plan._paths) > 512:
            plan._paths.clear()
            plan._paths[key] = hit
    nodes, children, edge_keys, getter = hit
    pslots, keep = _slot_matrix(engine, tmats, edge_keys, getter)
    lnl, snap = engine.eval(cache.snap, nodes, children, pslots, np.asarray(pi, dtype=np.float64),
                            want_snapshot=True, store_root=STORE_ROOT)
    return np.float64(lnl), PartialCache(engine, snap, site_map, cache.nodes())


def site_log_likelihoods(pi, root, ll_mats, edges, tmats, cache=None, categories=False):
    """Extension (no reference entry point): the per-column terms of lnL, for site-wise model comparison (WAIC,
    PSIS-LOO), site-rate estimates and site-wise tree tests.  Returns (lnL, site_lnl[n_columns], post or None) where
    lnL = sum(site_lnl) and, with categories, post[k, column] is the posterior probability of rate category k (equal
    category priors).  Arguments as for matML; with the PartialCache of this state only the root is recomputed (a
    LazyPartialCache not yet materialised, or no cache: one full pass that keeps nothing)."""
    refuse_sharded_site_lnl()
    engine, site_map = engine_for(ll_mats, len(tmats))
    plan = _plan_for(edges)
    if plan.nodes[-1] != root:
        raise KeyError(root)
    pi = np.asarray(pi, dtype=np.float64)
    if cache is not None and (not isinstance(cache, PartialCache) or cache.engine is not engine):
        raise TypeError("cache must be the cache returned by matML/cache_matML for this alignment")
    if cache is not None and not (isinstance(cache, LazyPartialCache) and cache._snap is None):
        kids = plan.kids[root]
        pslots, keep = _slot_matrix(engine, tmats, [(root, c) for c in kids])
        lnl, site, post, _ = engine.eval_sites(cache.snap, np.array([root], dtype=np.int32),
                                               np.array(kids, dtype=np.int32), pslots, pi, categories=categories)
    else:
        pslots, keep = _slot_matrix(engine, tmats, plan.edge_keys, plan=plan)
        lnl, site, post, _ = engine.eval_sites(None, plan.nodes, plan.children, pslots, pi, categories=categories)
    if site_map is not None:
        site = site[site_map]
        post = None if post is None else post[:, site_map]
    return np.float64(lnl), site, post


# --------------------------------------------------------- ML_gamma.pyx surface (Gamma rates)
def matML(pi, root, ll_mats, edges, tmats, n_sites, n_taxa, n_cats):
    """Full pruning pass over all rate categories (ML_gamma.pyx:7-42).  Returns (lnL, cache)."""
    return _full(pi, root, ll_mats, edges, tmats, len(tmats))


matML_cython = matML  # ML_gamma.pyx:44-79 is the same computation


def cache_matML(pi, root, ll_mats, cache_LL_Mats, nodes_recompute, edges, tmats, n_sites, n_taxa, n_cats):
    """Dirty-path pass: only `nodes_recompute` are recomputed, the rest comes from the cache
    (ML_gamma.pyx:83-118).  Returns (lnL, new cache); the input cache stays valid."""
    return _dirty(pi, root, ll_mats, cache_LL_Mats, nodes_recompute, edges, tmats, len(tmats))


def score_proposals(pi, root, ll_mats, cache_LL_Mats, proposals):
    """Extension (no reference entry point): lnL of many candidate proposals against one cache in
    a single launch.  `proposals` = iterable of (nodes_recompute, edges, tmats) as they would be
    passed to cache_matML.  Returns an array of lnL, one per candidate."""
    proposals = list(proposals)
    n_tables = len(proposals[0][2])
    engine, _ = engine_for(ll_mats, n_tables)
    if not isinstance(cache_LL_Mats, PartialCache) or cache_LL_Mats.engine is not engine:
        raise TypeError("cache must come from matML/cache_matML for this alignment")
    offsets, all_nodes, all_children, all_slots, keep_all = [0], [], [], [], []
    for nodes_recompute, edges, tmats in proposals:
        plan = _plan_for(edges)
        todo = sorted(set(nodes_recompute) | {root}, key=plan.index.__getitem__)
        edge_keys = [(n, c) for n in todo for c in plan.kids[n]]
        pslots, keep = _slot_matrix(engine, tmats, edge_keys)
        keep_all.append(keep)
        all_nodes.extend(todo)
        all_children.extend(c for n in todo for c in plan.kids[n])
        all_slots.append(pslots)
        offsets.append(len(all_nodes))
    return engine.eval_batch(cache_LL_Mats.snap, np.array(offsets, dtype=np.int32),
                             np.array(all_nodes, dtype=np.int32), np.array(all_children, dtype=np.int32),
                             np.ascontiguousarray(np.concatenate(all_slots, axis=0)),
                             np.asarray(pi, dtype=np.float64))


# ------------------------------------------------------------------ ML.pyx surface (one rate)
def matML_single(state, taxa, ll_mats):
    """ML.matML (ML.pyx:5-49): single rate category, arguments read from the state dict."""
    lnl, cache = _full(state["pi"], state["root"], ll_mats, state["postorder"], [state["transitionMat"]], 1)
    return lnl, cache


def cache_matML_single(state, taxa, ll_mats, cache_LL_Mat, nodes_recompute):
    """ML.cache_matML (ML.pyx:51-83)."""
    return _dirty(state["pi"], state["root"], ll_mats, cache_LL_Mat, nodes_recompute, state["postorder"],
                  [state["transitionMat"]], 1)
