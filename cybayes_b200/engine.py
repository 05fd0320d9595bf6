"""Device context of the likelihood engine: one alignment resident on one B200.

Thin, object-shaped wrapper over the C ABI (include/cybayes_b200.h).  Nothing here computes
likelihoods on the host; every number comes back from the CUDA library.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import numpy as np

from . import _lib
from ._lib import (CB_EVAL_FORCE_LEVELS, CB_EVAL_FORCE_WALK, CB_EVAL_NO_FOLD, CB_EVAL_NO_SYNC, CB_EVAL_STORE_ROOT, CB_EVAL_WANT_SNAPSHOT, c_f64p,
                   c_i32p, check)


def _f64(a):
    return a.ctypes.data_as(c_f64p)


def _i32(a):
    return a.ctypes.data_as(c_i32p)


class SlotBlock:
    """A run of consecutive P-matrix slots in the device pool, returned to the pool when the
    last table / handle referring to it is garbage collected."""
    __slots__ = ("_eng", "base", "n", "__weakref__")

    def __init__(self, eng, base, n):
        self._eng, self.base, self.n = eng, base, n

    def __del__(self):
        eng = self._eng
        if eng is not None and eng._ctx is not None:
            eng._free_slots.setdefault(self.n, []).append(self.base)


class SlotPool:
    """Id allocator for the P-matrix slot pool (ids are ours, storage is the backend's)."""

    def _init_slots(self):
        self._next_slot = 0
        self._reserved = 0
        self._free_slots = {}
        self._ctx = True

    def _reserve(self, n_slots):
        raise NotImplementedError

    def alloc_slots(self, n):
        free = self._free_slots.get(n)
        if free:
            base = free.pop()
        else:
            base = self._next_slot
            self._next_slot += n
            if self._next_slot > self._reserved:
                want = max(self._next_slot, 2 * self._reserved, 1024)
                self._reserve(want)
                self._reserved = want
        return SlotBlock(self, base, n)


class Engine(SlotPool):
    """codes: (n_taxa, n_patterns) uint8/uint16 state codes (see cb_set_tips); amb_sets: (n_amb, S)
    0/1 rows, row 0 all ones; weights: pattern multiplicities or None."""

    def __init__(self, codes, n_states, n_cats, amb_sets=None, weights=None, device=None):
        lib = _lib.load()
        self._lib = lib
        self._ctx = None
        codes = np.ascontiguousarray(codes)
        if codes.dtype not in (np.uint8, np.uint16):
            raise TypeError("codes must be uint8 or uint16")
        self.n_taxa, self.n_patterns = codes.shape
        self.n_states, self.n_cats = int(n_states), int(n_cats)
        self.code_dtype = codes.dtype
        if amb_sets is None:
            amb_sets = np.ones((1, n_states))
        amb_sets = np.ascontiguousarray(amb_sets, dtype=np.float64)
        if device is None:
            device = int(os.environ.get("CYBAYES_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        ctx = C.c_void_p()
        check(lib.cb_create(int(device), C.byref(ctx)))
        self._ctx = ctx
        self.device = int(device)
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        check(lib.cb_set_tips(ctx, self.n_taxa, self.n_patterns, self.n_states, self.n_cats,
                              codes.ctypes.data_as(C.c_void_p), codes.dtype.itemsize, _f64(amb_sets),
                              amb_sets.shape[0], None if w is None else _f64(w)))
        self.weights = w
        self._init_slots()
        self._ctx = ctx
        self._pending = []  # queued cb_pmat_build jobs
        self._lnl = np.zeros(1)
        self._snap = C.c_int(-1)
        self._state = {"alive": True}
        self._finalizer = weakref.finalize(self, Engine._destroy, lib, ctx, self._state)

    @staticmethod
    def _destroy(lib, ctx, state):
        state["alive"] = False   # handles that outlive the context (caches, slot blocks) become no-ops
        lib.cb_destroy(ctx)

    def close(self):
        if self._ctx is not None:
            self._finalizer()
            self._ctx = None

    # ------------------------------------------------------------------ multi-GPU
    @staticmethod
    def nccl_unique_id():
        buf = C.create_string_buffer(128)
        check(_lib.load().cb_nccl_unique_id(buf))
        return buf.raw

    def comm_init(self, unique_id, rank, n_ranks):
        check(self._lib.cb_comm_init(self._ctx, C.c_char_p(unique_id), int(rank), int(n_ranks)))

    # ------------------------------------------------------------------ P slots
    def _reserve(self, n_slots):
        check(self._lib.cb_pmat_reserve(self._ctx, n_slots))

    def upload_pmats(self, slots, mats):
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        mats = np.ascontiguousarray(mats, dtype=np.float64)
        assert mats.size == slots.size * self.n_states * self.n_states
        check(self._lib.cb_pmat_upload(self._ctx, slots.size, _i32(slots), _f64(mats)))

    def download_pmats(self, slots):
        self.flush_builds()
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        out = np.empty((slots.size, self.n_states, self.n_states))
        check(self._lib.cb_pmat_download(self._ctx, slots.size, _i32(slots), _f64(out)))
        return out

    def queue_build(self, model, pi, beta, gtr, slots, d, x=None):
        """Queue P(d) for `slots` (arrays or lists); consecutive jobs with the same model parameters
        are merged into ONE launch at the next evaluation (all branches x all rate categories)."""
        key = (model, float(beta), None if pi is None else pi.tobytes(), id(gtr), x is None)
        pend = self._pending
        if pend and pend[-1][0] == key:
            job = pend[-1]
            job[5].append(slots)
            job[6].append(d)
            if x is not None:
                job[7].append(x)
        else:
            pend.append([key, model, pi, float(beta), gtr, [slots], [d], [] if x is None else [x]])

    def flush_builds(self):
        pend = self._pending
        if not pend:
            return
        self._pending = []
        cat = np.concatenate
        for _, model, pi, beta, gtr, slots, d, x in pend:
            slots = np.ascontiguousarray(cat(slots) if len(slots) > 1 else slots[0], dtype=np.int32)
            d = np.ascontiguousarray(cat(d) if len(d) > 1 else d[0], dtype=np.float64)
            x_a = None if not x else np.ascontiguousarray(cat(x) if len(x) > 1 else x[0], dtype=np.float64)
            pi_a = None if pi is None else np.ascontiguousarray(pi, dtype=np.float64)
            check(self._lib.cb_pmat_build(self._ctx, int(model), None if pi_a is None else _f64(pi_a), beta,
                                          None if gtr is None else _f64(gtr), slots.size, _i32(slots), _f64(d),
                                          None if x_a is None else _f64(x_a)))

    # ------------------------------------------------------------------ evaluation
    def eval(self, snapshot, nodes, children, pslots, pi, want_snapshot=True, store_root=False,
             force_levels=False, sync=True, force_walk=False, no_fold=False):
        """Run the op list (see cb_eval).  Returns (lnL, snapshot id or -1)."""
        self.flush_builds()
        flags = (CB_EVAL_WANT_SNAPSHOT if want_snapshot else 0) | (CB_EVAL_STORE_ROOT if store_root else 0) \
            | (CB_EVAL_FORCE_LEVELS if force_levels else 0) | (0 if sync else CB_EVAL_NO_SYNC) \
            | (CB_EVAL_FORCE_WALK if force_walk else 0) | (CB_EVAL_NO_FOLD if no_fold else 0)
        pi = np.ascontiguousarray(pi, dtype=np.float64)
        check(self._lib.cb_eval(self._ctx, -1 if snapshot is None else int(snapshot), nodes.size, _i32(nodes),
                                _i32(children), _i32(pslots), _f64(pi), flags, C.byref(self._snap),
                                _f64(self._lnl)))
        return float(self._lnl[0]), int(self._snap.value)

    def eval_sites(self, snapshot, nodes, children, pslots, pi, want_snapshot=False, categories=False,
                   force_levels=False, force_walk=False, no_fold=False):
        """cb_eval with the per-pattern terms of lnL (see cb_eval_sites).  Returns (lnL, site_lnl[n_patterns],
        post[n_cats, n_patterns] -- the rate-category posteriors -- or None, snapshot id or -1)."""
        self.flush_builds()
        flags = (CB_EVAL_WANT_SNAPSHOT if want_snapshot else 0) | (CB_EVAL_FORCE_LEVELS if force_levels else 0) \
            | (CB_EVAL_FORCE_WALK if force_walk else 0) | (CB_EVAL_NO_FOLD if no_fold else 0)
        pi = np.ascontiguousarray(pi, dtype=np.float64)
        site = np.empty(self.n_patterns)
        post = np.empty((self.n_cats, self.n_patterns)) if categories else None
        check(self._lib.cb_eval_sites(self._ctx, -1 if snapshot is None else int(snapshot), nodes.size, _i32(nodes),
                                      _i32(children), _i32(pslots), _f64(pi), flags, C.byref(self._snap),
                                      _f64(self._lnl), _f64(site), None if post is None else _f64(post)))
        return float(self._lnl[0]), site, post, int(self._snap.value)

    def eval_batch(self, snapshot, offsets, nodes, children, pslots, pi):
        """Score many candidate dirty paths against one snapshot in a single launch."""
        self.flush_builds()
        offsets = np.ascontiguousarray(offsets, dtype=np.int32)
        out = np.empty(offsets.size - 1)
        pi = np.ascontiguousarray(pi, dtype=np.float64)
        check(self._lib.cb_eval_batch(self._ctx, -1 if snapshot is None else int(snapshot), offsets.size - 1,
                                      _i32(offsets), _i32(nodes), _i32(children), _i32(pslots), _f64(pi), _f64(out)))
        return out

    def simulate(self, parents, children, pslots, pi, root, seed, replicate, column_offset=0, download=True):
        """cb_simulate: overwrite every state cell of this context's alignment with a draw from the model (edges
        parents first, pslots[edge, category]).  Returns the replicate's codes (n_taxa, n_patterns), or None without
        download."""
        self.flush_builds()
        parents = np.ascontiguousarray(parents, dtype=np.int32)
        children = np.ascontiguousarray(children, dtype=np.int32)
        pslots = np.ascontiguousarray(pslots, dtype=np.int32)
        pi = np.ascontiguousarray(pi, dtype=np.float64)
        if not (parents.size == children.size and pslots.shape == (parents.size, self.n_cats) and pi.size == self.n_states):
            raise ValueError("parents, children, pslots (n_edges, n_cats) and pi (n_states) do not match")
        if not 0 <= int(replicate) < 1 << 32 or not 0 <= int(seed) < 1 << 64:
            raise ValueError("replicate must fit 32 bits and seed 64 bits, unsigned")
        out = np.empty((self.n_taxa, self.n_patterns), dtype=self.code_dtype) if download else None
        check(self._lib.cb_simulate(self._ctx, parents.size, _i32(parents), _i32(children), _i32(pslots), _f64(pi),
                                    int(root), int(seed), int(replicate), int(column_offset),
                                    None if out is None else out.ctypes.data_as(C.c_void_p)))
        return out

    def wait(self):
        check(self._lib.cb_result_wait(self._ctx, _f64(self._lnl)))
        return float(self._lnl[0])

    def retain_snapshot(self, snap):
        check(self._lib.cb_snapshot_retain(self._ctx, int(snap)))

    def release_snapshot(self, snap):
        if self._ctx is not None and self._state["alive"]:
            check(self._lib.cb_snapshot_release(self._ctx, int(snap)))

    def read_partial(self, snap, node, with_scale=False):
        """(C, S, n_patterns) partial of `node`; unscaled like the reference's cache entries unless
        with_scale, in which case (mantissas, per-pattern exponents) is returned."""
        out = np.empty((self.n_cats, self.n_states, self.n_patterns))
        if with_scale:
            sc = np.empty(self.n_patterns, dtype=np.int32)
            check(self._lib.cb_snapshot_read(self._ctx, int(snap), int(node), _f64(out), _i32(sc)))
            return out, sc
        check(self._lib.cb_snapshot_read(self._ctx, int(snap), int(node), _f64(out), None))
        return out

    # ------------------------------------------------------------------ measurement
    def stats(self):
        v = [C.c_int64() for _ in range(4)]
        check(self._lib.cb_stats(self._ctx, *[C.byref(x) for x in v]))
        return {"kernel_launches": v[0].value, "h2d_bytes": v[1].value, "d2h_bytes": v[2].value,
                "device_bytes": v[3].value}

    def mem_info(self):
        """Device memory as the context sees it: free / total bytes, bytes pooled in unused partial buffers, bytes of
        one partial buffer."""
        x = [C.c_int64() for _ in range(4)]
        check(self._lib.cb_mem_info(self._ctx, *[C.byref(t) for t in x]))
        return {"free": x[0].value, "total": x[1].value, "pooled": x[2].value, "partial": x[3].value}

    def last_eval_ms(self):
        ms = C.c_float()
        check(self._lib.cb_last_eval_ms(self._ctx, C.byref(ms)))
        return float(ms.value)

    def last_eval_main_ms(self):
        """Device time of the pruning launches alone (no P-layout / op-image pre-pass)."""
        ms = C.c_float()
        check(self._lib.cb_last_eval_main_ms(self._ctx, C.byref(ms)))
        return float(ms.value)

    def last_eval_info(self):
        """What the last evaluation had to move (bytes, from its op list) and how it was scheduled."""
        w, r = C.c_int64(), C.c_int64()
        counts = np.zeros(8, dtype=np.int32)
        check(self._lib.cb_last_eval_info(self._ctx, C.byref(w), C.byref(r), _i32(counts)))
        names = ("ops", "stored", "read_back", "stack_pops", "spills", "cherries_folded", "launches", "small_records")
        out = dict(zip(names, (int(x) for x in counts)))
        out["bytes_written"], out["bytes_read"] = w.value, r.value
        return out

    def host_profile(self, reset=True):
        """Mean host microseconds per evaluation call since the last reset, by phase."""
        a = np.zeros(6)
        check(self._lib.cb_host_profile(self._ctx, _f64(a), 1 if reset else 0))
        n = max(a[5], 1.0)
        return {"plan": a[0] / n, "fill": a[1] / n, "upload_launch": a[2] / n, "wait": a[3] / n, "bookkeeping": a[4] / n,
                "calls": int(a[5])}

    def mark(self, which):
        check(self._lib.cb_mark(self._ctx, int(which)))

    def mark_elapsed_ms(self):
        ms = C.c_float()
        check(self._lib.cb_mark_elapsed_ms(self._ctx, C.byref(ms)))
        return float(ms.value)

    def sync(self):
        check(self._lib.cb_sync(self._ctx))

    def fp64_peak_tflops(self):
        """FP64 tensor-core peak of this GPU measured from registers (roofline denominator for S = 64)."""
        out = np.zeros(1)
        check(self._lib.cb_fp64_peak(self._ctx, _f64(out)))
        return float(out[0])

    def flush_l2(self):
        check(self._lib.cb_flush_l2(self._ctx))
