"""MCMC with the generation loop inside the library (SURVEY 8f rank 1).

``run_chain_native`` is ``driver.run_chain`` with the Metropolis-Hastings loop moved out of the interpreter:
the start state is drawn in Python exactly as the reference does (state_init, both generators seeded with the
driver's seed), the two Mersenne-Twister states are handed to ``cb_chain_*`` (csrc/mcmc_native.cuh), and every
``thin`` generations control comes back for the ``.log`` / ``.trees`` / stdout lines.  For a fixed seed the chain
takes the moves and the accept / reject decisions of the reference driver generation by generation (the recorded
traces of tests/golden pin this, on the GPU and -- through an oracle-backed backend -- on CPU).

External-SPR proposals are scored by their two dirty paths (the reference runs a full pass,
mat_mcmc_gamma.py:167-169); the numbers are bit-identical because the same kernels see the same operands.
"""
from __future__ import annotations

import ctypes as C
import random
import sys
import time

import numpy as np

from . import _lib, config, likelihood, subst
from ._lib import c_f64p, c_i32p
from .driver import load_alignment, move_table, open_site_lnl, write_site_lnl
from .mcmc_gamma import adjlist2newickBL, adjlist2nodes_dict, get_siterates, state_init

MOVES = [("bl", "scale_edge"), ("bl", "node_slider"), ("tree", "rooted_NNI"), ("tree", "externalSPR"),
         ("pi", "mvDualSlider"), ("srates", "scale_alpha"), ("rates", "mvDualSlider")]
PARAM_IDS = {"pi": 0, "rates": 1, "tree": 2, "bl": 3, "srates": 4}
MODEL_IDS = {"JC": 0, "F81": 1, "GTR": 2}

_BUILD_FN, _EVAL_FN, _RELEASE_FN = _lib.CHAIN_BUILD_FN, _lib.CHAIN_EVAL_FN, _lib.CHAIN_RELEASE_FN
_RATES_FN, _BETA_FN, _EIG_FN = _lib.CHAIN_RATES_FN, _lib.CHAIN_BETA_FN, _lib.CHAIN_EIG_FN
_EVAL_SITES_FN = _lib.CHAIN_EVAL_SITES_FN
ChainBackend = _lib.ChainBackend


def _host_callbacks(n_states, n_cats, n_rates):
    """The three host functions whose bits depend on SciPy / BLAS, as ctypes callbacks."""
    def rates_cb(_user, alpha, out):
        try:
            r = get_siterates(alpha)
            for k in range(n_cats):
                out[k] = r[k]
            return 0
        except Exception:
            return 1

    def beta_cb(_user, pi, n, out):
        try:
            out[0] = subst.f81_beta(np.ctypeslib.as_array(pi, shape=(n,)).copy())
            return 0
        except Exception:
            return 1

    def eig_cb(_user, pi, er, out):
        try:
            eig = subst.gtr_eigensystem(np.ctypeslib.as_array(pi, shape=(n_states,)).copy(),
                                        np.ctypeslib.as_array(er, shape=(n_rates,)).copy())
            C.memmove(out, eig.ctypes.data, eig.nbytes)
            return 0
        except Exception:
            return 1
    return _RATES_FN(rates_cb), _BETA_FN(beta_cb), _EIG_FN(eig_cb)


def engine_callbacks(engine):
    """Evaluation backend over any object with the Engine methods (the CPU tests pass the oracle-backed fake):
    (pmat_build, eval, snapshot_release, eval_sites) as ctypes callbacks."""
    S, Cc = engine.n_states, engine.n_cats

    def build_cb(_user, model, pi, beta, gtr, count, slots, d, x):
        try:
            pi_a = np.ctypeslib.as_array(pi, shape=(S,)).copy()
            gtr_a = np.ctypeslib.as_array(gtr, shape=(S + 2 * S * S,)).copy() if gtr else None
            engine.queue_build(model, pi_a, beta, gtr_a, np.ctypeslib.as_array(slots, shape=(count,)).copy(),
                               np.ctypeslib.as_array(d, shape=(count,)).copy(),
                               np.ctypeslib.as_array(x, shape=(count,)).copy() if x else None)
            return 0
        except Exception:
            import traceback
            traceback.print_exc()
            return 1

    def eval_cb(_user, snap_in, n_ops, nodes, children, pslots, pi, flags, snap_out, lnl_out):
        try:
            lnl, snap = engine.eval(None if snap_in < 0 else snap_in, np.ctypeslib.as_array(nodes, shape=(n_ops,)).copy(),
                                    np.ctypeslib.as_array(children, shape=(2 * n_ops,)).copy(),
                                    np.ctypeslib.as_array(pslots, shape=(2 * n_ops, Cc)).copy(),
                                    np.ctypeslib.as_array(pi, shape=(S,)).copy(), want_snapshot=bool(flags & 1))
            snap_out[0] = snap
            lnl_out[0] = lnl
            return 0
        except Exception:
            import traceback
            traceback.print_exc()
            return 1

    def release_cb(_user, snap):
        engine.release_snapshot(snap)
        return 0

    def eval_sites_cb(_user, snap_in, n_ops, nodes, children, pslots, pi, flags, snap_out, lnl_out, site_out, post_out):
        try:
            lnl, site, post, snap = engine.eval_sites(
                None if snap_in < 0 else snap_in, np.ctypeslib.as_array(nodes, shape=(n_ops,)).copy(),
                np.ctypeslib.as_array(children, shape=(2 * n_ops,)).copy(),
                np.ctypeslib.as_array(pslots, shape=(2 * n_ops, Cc)).copy(), np.ctypeslib.as_array(pi, shape=(S,)).copy(),
                want_snapshot=bool(flags & 1), categories=bool(post_out))
            P = engine.n_patterns
            np.ctypeslib.as_array(site_out, shape=(P,))[:] = site
            if post_out:
                np.ctypeslib.as_array(post_out, shape=(Cc, P))[:] = post
            snap_out[0] = snap
            lnl_out[0] = lnl
            return 0
        except Exception:
            import traceback
            traceback.print_exc()
            return 1
    return _BUILD_FN(build_cb), _EVAL_FN(eval_cb), _RELEASE_FN(release_cb), _EVAL_SITES_FN(eval_sites_cb)


class NativeChain:
    """Thin object over cb_chain_*; the start state comes from Python, generations run in the library."""

    def __init__(self, engine, state, site_rates, model, binary, use_callbacks=False, skip_degenerate_rates=False,
                 site_map=None):
        lib = _lib.load()
        self._lib, self.engine, self._site_map = lib, engine, site_map
        self.n_taxa, self.n_states, self.n_cats = config.N_TAXA, engine.n_states, engine.n_cats
        tree = state["tree"]
        self.n_edges = len(tree)
        n_rates = len(state["rates"])
        params, weights, _, tree_w, bl_w = move_table(model, n_rates, skip_degenerate_rates)
        cdf = np.ascontiguousarray(np.cumsum(weights) / np.sum(weights))
        tree_cdf = np.ascontiguousarray(np.cumsum(tree_w) / np.sum(tree_w))
        bl_cdf = np.ascontiguousarray(np.cumsum(bl_w) / np.sum(bl_w))
        ids = np.array([PARAM_IDS[p] for p in params], dtype=np.int32)
        self._host = _host_callbacks(self.n_states, self.n_cats, n_rates)
        be = ChainBackend()
        be.site_rates, be.f81_beta, be.gtr_eig = self._host
        ctx = None
        if use_callbacks or not hasattr(engine, "_ctx") or not isinstance(engine._ctx, C.c_void_p):
            self._eng_cbs = engine_callbacks(engine)
            be.pmat_build, be.eval, be.snapshot_release, be.eval_sites = self._eng_cbs
        else:
            engine.flush_builds()
            ctx = engine._ctx
        n_slots = 2 * self.n_edges * self.n_cats + 16 * self.n_cats
        self._block = engine.alloc_slots(n_slots)
        self._chain = C.c_void_p()
        _lib.check(lib.cb_chain_create(ctx, C.byref(be), self.n_taxa, self.n_states, self.n_cats, MODEL_IDS[model],
                                       1 if binary else 0, int(state["root"]), self._block.base, n_slots, subst.HOST_EXP_MAX,
                                       len(ids), ids.ctypes.data_as(c_i32p), cdf.ctypes.data_as(c_f64p),
                                       tree_cdf.ctypes.data_as(c_f64p), bl_cdf.ctypes.data_as(c_f64p), C.byref(self._chain)))
        self._be = be
        parents = np.array([p for p, _ in tree], dtype=np.int32)
        children = np.array([c for _, c in tree], dtype=np.int32)
        lengths = np.array(list(tree.values()), dtype=np.float64)
        pi = np.ascontiguousarray(state["pi"], dtype=np.float64)
        rates = np.ascontiguousarray(state["rates"], dtype=np.float64)
        sr = np.ascontiguousarray(site_rates, dtype=np.float64)
        beta = float(config.NORM_BETA)
        if model == "F81":
            beta = float(subst.f81_beta(pi))
        eig = subst.gtr_eigensystem(pi, rates) if model == "GTR" else None
        lnl = C.c_double()
        _lib.check(lib.cb_chain_set_state(self._chain, self.n_edges, parents.ctypes.data_as(c_i32p),
                                          children.ctypes.data_as(c_i32p), lengths.ctypes.data_as(c_f64p),
                                          pi.ctypes.data_as(c_f64p), n_rates, rates.ctypes.data_as(c_f64p),
                                          float(state["srates"]), sr.ctypes.data_as(c_f64p), beta,
                                          None if eig is None else eig.ctypes.data_as(c_f64p), C.byref(lnl)))
        self.initial_lnl = lnl.value
        self.n_rates = n_rates

    def take_rng(self):
        """Hand the interpreter's two Mersenne-Twister states to the chain."""
        _, st, _ = random.getstate()
        py = np.array(st[:624], dtype=np.uint32)
        key = np.random.get_state(legacy=True)
        npk = np.ascontiguousarray(key[1], dtype=np.uint32)
        u32p = C.POINTER(C.c_uint32)
        _lib.check(self._lib.cb_chain_set_rng(self._chain, py.ctypes.data_as(u32p), int(st[624]), npk.ctypes.data_as(u32p),
                                              int(key[2])))

    def give_rng(self):
        """... and back (the interpreter continues the streams where the chain left them)."""
        py, npk = np.zeros(624, dtype=np.uint32), np.zeros(624, dtype=np.uint32)
        p1, p2 = C.c_int(), C.c_int()
        u32p = C.POINTER(C.c_uint32)
        _lib.check(self._lib.cb_chain_get_rng(self._chain, py.ctypes.data_as(u32p), C.byref(p1), npk.ctypes.data_as(u32p),
                                              C.byref(p2)))
        random.setstate((3, tuple(int(x) for x in py) + (p1.value,), None))
        np.random.set_state(("MT19937", npk, p2.value, 0, 0.0))

    def run(self, n, trace=True):
        i8p = C.POINTER(C.c_int8)
        if trace:
            mv, acc = np.zeros(n, dtype=np.int8), np.zeros(n, dtype=np.int8)
            cur, prop, ratio, logu = (np.zeros(n) for _ in range(4))
            _lib.check(self._lib.cb_chain_run(self._chain, n, mv.ctypes.data_as(i8p), acc.ctypes.data_as(i8p),
                                              cur.ctypes.data_as(c_f64p), prop.ctypes.data_as(c_f64p),
                                              ratio.ctypes.data_as(c_f64p), logu.ctypes.data_as(c_f64p)))
            return mv, acc, cur, prop, ratio, logu
        _lib.check(self._lib.cb_chain_run(self._chain, n, None, None, None, None, None, None))
        return None

    def state(self):
        E = self.n_edges
        parents, children = np.zeros(E, dtype=np.int32), np.zeros(E, dtype=np.int32)
        lengths, pi, rates = np.zeros(E), np.zeros(self.n_states), np.zeros(self.n_rates)
        sr = np.zeros(self.n_cats)
        alpha, lnl = C.c_double(), C.c_double()
        _lib.check(self._lib.cb_chain_get_state(self._chain, parents.ctypes.data_as(c_i32p), children.ctypes.data_as(c_i32p),
                                                lengths.ctypes.data_as(c_f64p), pi.ctypes.data_as(c_f64p),
                                                rates.ctypes.data_as(c_f64p), C.byref(alpha), sr.ctypes.data_as(c_f64p),
                                                C.byref(lnl)))
        tree = {(int(p), int(c)): float(t) for p, c, t in zip(parents, children, lengths)}
        return {"tree": tree, "pi": pi, "rates": rates, "srates": alpha.value, "site_rates": sr.tolist(),
                "logLikehood": np.float64(lnl.value)}

    def site_lnl(self, categories=False):
        """Per-column terms of the current state's lnL (cb_chain_site_lnl), in alignment-column order when the engine
        holds compressed patterns (`site_map`), and with categories the (n_cats, columns) rate-category posteriors.
        Returns (site_lnl, post or None).  Takes no random draw."""
        P = self.engine.n_patterns
        site = np.empty(P)
        post = np.empty((self.n_cats, P)) if categories else None
        _lib.check(self._lib.cb_chain_site_lnl(self._chain, site.ctypes.data_as(c_f64p),
                                               None if post is None else post.ctypes.data_as(c_f64p)))
        if self._site_map is not None:
            site = site[self._site_map]
            post = None if post is None else post[:, self._site_map]
        return site, post

    def counters(self):
        m, a = np.zeros(7, dtype=np.int64), np.zeros(7, dtype=np.int64)
        i64p = C.POINTER(C.c_int64)
        _lib.check(self._lib.cb_chain_counters(self._chain, m.ctypes.data_as(i64p), a.ctypes.data_as(i64p)))
        return m, a

    def close(self):
        if self._chain:
            self._lib.cb_chain_destroy(self._chain)
            self._chain = C.c_void_p()

    def __del__(self):
        try:
            if self.engine._ctx is not None:
                self.close()
        except Exception:
            pass


def run_chain_native(input_file, model, n_gen, thin, data_type, output_file, reader=None, seed=1234, out=sys.stdout,
                     on_generation=None, diag=None, use_callbacks=False, skip_degenerate_rates=False, site_lnl=False, ppc=0, ppc_seed=1):
    """driver.run_chain with the generation loop in the library; same files, same stdout, same return value.
    site_lnl: also write <output_file>.sitelnl (driver.run_chain), from cb_chain_site_lnl at every sample.
    ppc, ppc_seed: also write <output_file>.ppc (driver.run_chain), from NativeChain.state() at every sample."""
    if site_lnl:
        likelihood.refuse_sharded_site_lnl()
    if ppc:
        from .ppc import refuse_sharded_ppc
        refuse_sharded_ppc()
    np.random.seed(seed)
    random.seed(seed)
    load_alignment(input_file, data_type, reader)
    config.N_GEN, config.THIN, config.MODEL = n_gen, thin, model
    print("Characters ", config.N_CHARS, file=out)
    print("TAXA ", config.TAXA, file=out)
    print("Number of TAXA ", config.N_TAXA, file=out)
    print("Alphabet ", config.ALPHABET, file=out)
    if model == "JC":
        config.NORM_BETA = config.N_CHARS / (config.N_CHARS - 1)  # overwritten by state_init (:580)
    state = state_init()
    site_rates = get_siterates(state["srates"])
    root = state["root"]
    engine, site_map = likelihood.engine_for(config.LEAF_LLMAT, config.N_CATS)
    chain = NativeChain(engine, state, site_rates, model, config.IN_DTYPE == "bin", use_callbacks=use_callbacks,
                        skip_degenerate_rates=skip_degenerate_rates, site_map=site_map)
    state["logLikehood"] = np.float64(chain.initial_lnl)
    print("Initial Random Tree ", adjlist2newickBL(state["tree"], adjlist2nodes_dict(state["tree"]), root) + ";",
          sep="\t", file=out)
    print("Initial Likelihood ", state["logLikehood"], file=out)
    initial_lnl = state["logLikehood"]
    log_fh = open(output_file + ".log", "w")
    trees_fh = open(output_file + ".trees", "w")
    print("Iter", "LnL", "TL", "Alpha", sep="\t", file=log_fh)
    site_fh = open_site_lnl(output_file, config.N_SITES) if site_lnl else None
    reps = ppc_fh = None
    if ppc:
        from .ppc import Replicates, open_ppc, write_sample
        reps, ppc_fh = Replicates(config.LEAF_LLMAT, config.N_CATS), open_ppc(output_file)
    chain.take_rng()
    first_seen = {}
    want_trace = True
    t_start = time.perf_counter()
    done = 0
    while done < n_gen:
        n = min(thin - done % thin, n_gen - done)
        mv, acc, cur, prop, ratio, logu = chain.run(n, trace=want_trace)
        for m in np.unique(mv):
            first_seen.setdefault(int(m), done + int(np.argmax(mv == m)))
        if on_generation is not None:
            for j in range(n):
                if diag is not None:
                    diag["ll_ratio"], diag["log_u"] = float(ratio[j]), float(logu[j])
                p, name = MOVES[mv[j]]
                on_generation(done + j + 1, np.float64(cur[j]), np.float64(prop[j]), p, name, bool(acc[j]), None)
        done += n
        if done % thin == 0:
            st = chain.state()
            TL = sum(st["tree"].values())
            sampled = adjlist2newickBL(st["tree"], adjlist2nodes_dict(st["tree"]), root) + ";"
            p, name = MOVES[mv[-1]]
            print(done, np.float64(cur[-1]), np.float64(prop[-1]), TL, p, name, sep="\t", file=out)
            print(done, st["logLikehood"], TL, st["srates"], sep="\t", file=log_fh)
            print(done, sampled, sep="\t", file=trees_fh)
            if site_fh is not None:
                write_site_lnl(site_fh, done, chain.site_lnl()[0])
            if reps is not None:
                st["root"] = root
                write_sample(ppc_fh, reps, done, done // thin - 1, st, model, ppc, ppc_seed)
    elapsed = time.perf_counter() - t_start
    chain.give_rng()
    log_fh.close()
    trees_fh.close()
    if site_fh is not None:
        site_fh.close()
    if reps is not None:
        ppc_fh.close()
        reps.close()
    final = chain.state()
    final["root"] = root
    m, a = chain.counters()
    moves_count, accepts_count = {}, {}
    for mid in sorted(first_seen, key=first_seen.get):
        moves_count[MOVES[mid]] = int(m[mid])
        accepts_count[MOVES[mid]] = int(a[mid])
    for k, v in moves_count.items():
        print(k, accepts_count[k], v, file=out)
    chain.close()
    return {"state": final, "initial_lnL": initial_lnl, "moves": moves_count, "accepts": accepts_count,
            "seconds": elapsed, "gens_per_sec": n_gen / elapsed if elapsed > 0 else float("inf")}
