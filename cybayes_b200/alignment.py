"""Phylip readers, leaf encoding and site-pattern compression (host side).

Restates utils.pyx:11-120.  The reference materialises one (S, P) float64 0/1 matrix per
taxon (``sites2Mat``); here the alignment is kept as compact integer *state codes*
(1 byte per cell for up to ~250 states) -- that is what the GPU reads -- and the float
matrices of the reference contract are produced on demand by ``LeafMatrices``.

Code convention (shared with cb_set_tips): ``code < S`` is that state; ``code = S + k`` is the
k-th ambiguity set, set 0 being the all-ones column of '?' / '-' (utils.pyx:99-100), later
sets the 'a/b' multi-hot columns (utils.pyx:102-106) in order of first appearance.
"""
from __future__ import annotations

import os

import numpy as np

# the reference pins BLAS threading at import of utils (utils.pyx:3-7); kept for parity of
# whatever NumPy work the caller still does on the host
for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "VECLIB_MAXIMUM_THREADS",
           "NUMEXPR_NUM_THREADS"):
    os.environ[_v] = "1"

MISSING = ("?", "-")


class LeafMatrices(dict):
    """``config.LEAF_LLMAT``: mapping 1-based taxon id -> (S, P) float64 0/1 matrix, exactly the
    objects ``sites2Mat`` returns (utils.pyx:94-120), but backed by integer codes and
    materialised lazily (a 1024 x 1M binary alignment is 1 GB of codes, 16 GB of matrices)."""

    def __init__(self, codes, n_states, amb_sets):
        super().__init__()
        self.codes = codes                # (n_taxa, n_sites) uint8 / uint16
        self.n_states = int(n_states)
        self.amb_sets = amb_sets          # (n_amb, S) float64, row 0 = all ones
        self._ids = range(1, codes.shape[0] + 1)

    def __missing__(self, key):
        if key not in self._ids:
            raise KeyError(key)
        mat = self.dense(key)
        self[key] = mat
        return mat

    def dense(self, key):
        S = self.n_states
        row = self.codes[key - 1].astype(np.int64)
        table = np.vstack([np.eye(S), self.amb_sets])  # code -> column
        return np.ascontiguousarray(table[row].T)

    # a dict that lazily fills must still look complete to callers that iterate
    def keys(self):
        return self._ids

    def __iter__(self):
        return iter(self._ids)

    def __len__(self):
        return len(self._ids)

    def __contains__(self, key):
        return key in self._ids

    def items(self):
        return ((k, self[k]) for k in self._ids)

    def values(self):
        return (self[k] for k in self._ids)


def encode_tokens(rows, alphabet):
    """rows: list (taxon order) of token sequences.  Returns (codes, amb_sets)."""
    S = len(alphabet)
    index = {a: i for i, a in enumerate(alphabet)}
    amb_index = {}
    amb_rows = [np.ones(S)]
    n_taxa, n_sites = len(rows), len(rows[0])
    lookup = dict(index)
    for m in MISSING:
        lookup[m] = S
    wide = np.empty((n_taxa, n_sites), dtype=np.int64)
    # single-character alphabets (binary / readMultiPhy rows given as strings): one table lookup per row
    lut = None
    if all(len(a) == 1 and ord(a) < 256 for a in alphabet):
        lut = np.full(256, -1, dtype=np.int64)
        for a, i in index.items():
            lut[ord(a)] = i
        for m in MISSING:
            lut[ord(m)] = S
    for t, toks in enumerate(rows):
        if len(toks) != n_sites:
            raise ValueError(f"taxon {t + 1}: {len(toks)} characters, expected {n_sites}")
        if lut is not None:
            codes_row = None
            try:
                text = toks if isinstance(toks, str) else "".join(toks)
                if len(text) == n_sites:  # every token is one character
                    codes_row = lut[np.frombuffer(text.encode("latin-1"), dtype=np.uint8)]
            except (UnicodeEncodeError, TypeError):
                codes_row = None
            if codes_row is not None and (codes_row >= 0).all():
                wide[t] = codes_row
                continue
        try:
            wide[t] = [lookup[tok] for tok in toks]
        except KeyError:
            for p, tok in enumerate(toks):
                code = lookup.get(tok)
                if code is None:
                    if "/" not in tok:
                        raise ValueError(f"{tok!r} is not in list")  # alphabet.index(...) in utils.pyx:110
                    members = tuple(sorted({index[x] for x in tok.split("/")}))
                    if len(members) == S:
                        code = S
                    else:
                        if members not in amb_index:
                            amb_index[members] = len(amb_rows)
                            v = np.zeros(S)
                            v[list(members)] = 1.0
                            amb_rows.append(v)
                        code = S + amb_index[members]
                    lookup[tok] = code
                wide[t, p] = code
    n_codes = S + len(amb_rows)
    dtype = np.uint8 if n_codes <= 256 else np.uint16
    if n_codes > 65536:
        raise ValueError("too many states / ambiguity sets")
    return wide.astype(dtype), np.array(amb_rows)


def sites2Mat(sites, n_chars, alphabet, taxa_list):
    """Leaf encoding (utils.pyx:94-120): taxon id = position in `taxa_list` + 1."""
    rows = [sites[name] for name in taxa_list]
    codes, amb = encode_tokens(rows, alphabet)
    return LeafMatrices(codes, n_chars, amb)


def _read(fname, mode):
    site_dict, alphabet, taxa_list = {}, [], []
    if mode == "binary":
        alphabet = ["0", "1"]  # utils.pyx:21
    with open(fname) as fh:
        header = fh.readline().strip()
        n_leaves, n_sites = map(int, header.split(" "))
        for line in fh:
            line = line.strip()
            if len(line) < 1:
                continue
            if mode == "tokens":
                taxon, vec = line.split("\t")
                chars = vec.split(" ")
                seen = [t for tok in chars for t in tok.split("/")]
            else:
                fields = line.split()
                if len(fields) != 2:
                    if mode == "multi" and "\t" in line:
                        # extension: tab + space-separated tokens is the readPhy layout; the
                        # reference's readMultiPhy raises here (utils.pyx:78, SURVEY F4)
                        taxon, vec = line.split("\t")
                        chars = vec.split(" ")
                        seen = [t for tok in chars for t in tok.split("/")]
                        fields = None
                    else:
                        raise ValueError("too many values to unpack (expected 2)" if len(fields) > 2
                                         else f"not enough values to unpack (expected 2, got {len(fields)})")
                if fields is not None:
                    taxon, vec = fields
                    if mode == "binary":
                        assert len(vec) == n_sites
                        chars = vec
                    else:
                        chars = list(vec)
                    seen = vec
            taxon = taxon.replace(" ", "")
            for ch in dict.fromkeys(seen):  # distinct symbols in order of first appearance
                if ch not in alphabet and ch not in MISSING:
                    alphabet.append(ch)
            site_dict[taxon] = chars
            taxa_list.append(taxon)
    n_chars = len(alphabet)
    ll_mats = sites2Mat(site_dict, n_chars, alphabet, taxa_list)
    return n_leaves, n_chars, alphabet, site_dict, ll_mats, taxa_list, n_sites


def readBinaryPhy(fname):
    """'name 0101?...' rows; alphabet pre-seeded with '0','1' (utils.pyx:11-37)."""
    return _read(fname, "binary")


def readPhy(fname):
    """'name<TAB>tok tok tok' rows, '/' separates polymorphic states (utils.pyx:39-65).
    (The reference also prints every row; that debugging output is not reproduced.)"""
    return _read(fname, "tokens")


def readMultiPhy(fname):
    """'name CHARS' rows, one character per site (utils.pyx:67-92)."""
    return _read(fname, "multi")


# ----------------------------------------------------------------------------- patterns
def compress_patterns(codes):
    """Unique alignment columns in order of first appearance.

    Returns (pattern_codes (n_taxa, n_patterns), weights (n_patterns,) float64,
    site_to_pattern (n_sites,) int64).  The reference evaluates every column (SURVEY F2);
    summing weight * log-likelihood over unique columns is the same number up to summation
    order."""
    n_taxa, n_sites = codes.shape
    cols = np.ascontiguousarray(codes.T)
    keys = cols.view(np.dtype((np.void, cols.dtype.itemsize * n_taxa))).ravel()
    _, first, inverse, counts = np.unique(keys, return_index=True, return_inverse=True, return_counts=True)
    order = np.argsort(first, kind="stable")          # sorted-unique index -> first-appearance rank
    rank = np.empty_like(order)
    rank[order] = np.arange(order.size)
    pattern_codes = np.ascontiguousarray(cols[first[order]].T)
    return pattern_codes, counts[order].astype(np.float64), rank[inverse.ravel()]


def compress_patterns_gpu(codes, device=None):
    """compress_patterns for alignments too long for the host route (10^5 .. 10^7 columns): the column comparison runs
    on the GPU (cb_compress_patterns: 128-bit column hashes, verified column by column, so the result is exact).
    Same return value as compress_patterns, element for element."""
    codes = np.ascontiguousarray(codes)
    weights, site_to_pattern, first = pattern_weights_gpu(codes, device)
    return np.ascontiguousarray(codes[:, first]), weights, site_to_pattern


def pattern_weights_gpu(codes, device=None):
    """compress_patterns_gpu without gathering the pattern columns: (weights, site_to_pattern, first_site) -- what a
    statistic of the column multiplicities needs."""
    import ctypes as C

    from . import _lib
    lib = _lib.load()
    codes = np.ascontiguousarray(codes)
    n_taxa, n_sites = codes.shape
    if device is None:
        device = int(os.environ.get("CYBAYES_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    site_to_pattern = np.empty(n_sites, dtype=np.int64)
    first = np.empty(n_sites, dtype=np.int64)
    weights = np.empty(n_sites, dtype=np.float64)
    n_pat = C.c_int64()
    _lib.check(lib.cb_compress_patterns(int(device), codes.ctypes.data_as(C.c_void_p), n_taxa, n_sites, codes.dtype.itemsize,
                                        site_to_pattern.ctypes.data_as(_lib.c_i64p), first.ctypes.data_as(_lib.c_i64p),
                                        weights.ctypes.data_as(_lib.c_f64p), C.byref(n_pat)))
    n = n_pat.value
    return weights[:n].copy(), site_to_pattern, first[:n].copy()
