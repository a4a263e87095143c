"""Held-out pairs for choosing K by held-out likelihood (BigCLAM, Yang & Leskovec; the thesis p.20).

split_pairs() leaves out a fraction of the node pairs: as many non-adjacent pairs as edges, so that both terms of the
objective are scored.  The solver is then fitted on the remaining pairs with the masked objective (BigClam.set_holdout,
bigclam_set_holdout in the C ABI), and BigClam.holdout_loglikelihood() scores the left-out pairs
(BigClam.select_K does the whole loop).  The split is pure NumPy host code; the fit and the scoring run on the GPU.
"""
from __future__ import annotations

from typing import NamedTuple

import numpy as np


class Split(NamedTuple):
    rowptr: np.ndarray        # training graph (CSR, int64 / int32): E minus the held-out edges, list order kept
    col: np.ndarray
    ho_rowptr: np.ndarray     # held-out pairs, both directions, ascending partners per node
    ho_col: np.ndarray
    ho_is_edge: np.ndarray    # uint8 per held-out entry: 1 = held-out edge, 0 = held-out non-edge


def _check_simple(rowptr, col):
    n = len(rowptr) - 1
    u = np.repeat(np.arange(n, dtype=np.int64), np.diff(rowptr))
    v = col.astype(np.int64)
    if (u == v).any():
        raise ValueError("split_pairs needs a simple graph: self loop found (read the edge list with multiplicity='dedup')")
    key = u * n + v
    if len(np.unique(key)) != len(key):
        raise ValueError("split_pairs needs a simple graph: repeated neighbour found (read the edge list with multiplicity='dedup')")
    if not np.array_equal(np.sort(key), np.sort(v * n + u)):
        raise ValueError("split_pairs needs a simple graph: the neighbour lists are not symmetric")
    return n, u, v


def _csr(n, a, b, *vals):
    order = np.lexsort((b, a))
    rowptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(a, minlength=n), out=rowptr[1:])
    return (rowptr, b[order].astype(np.int32), *(x[order] for x in vals))


def split_pairs(rowptr, col, ho_frac: float = 0.2, seed: int = 0) -> Split:
    """Holds out exactly round(ho_frac |E|) undirected edges, drawn without replacement, and as many distinct
    non-adjacent pairs, drawn uniformly without replacement.  Randomness: numpy.random.Generator(PCG64(seed)), so a given
    graph, fraction and seed always give the same split.  Raises ValueError for a graph that is not simple (self loops,
    repeated or one-sided neighbours): with literal multiplicity a held-out edge would stay in training as its duplicate."""
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int64)
    col = np.ascontiguousarray(col, dtype=np.int32)
    if not 0.0 <= ho_frac < 1.0:
        raise ValueError("ho_frac must be in [0, 1)")
    n, u, v = _check_simple(rowptr, col)
    up = u < v
    eu, ev = u[up], v[up]                                  # every undirected edge once, in CSR order
    m = len(eu)
    h = int(round(ho_frac * m))
    if h > n * (n - 1) // 2 - m:
        raise ValueError("split_pairs: not enough non-adjacent pairs to hold out")
    rng = np.random.Generator(np.random.PCG64(seed))
    pick = np.sort(rng.choice(m, size=h, replace=False)) if h > 0 else np.zeros(0, dtype=np.int64)
    ho_e_key = np.sort(eu[pick] * n + ev[pick])
    # non-edges: uniform ordered pairs u != v by rejection, unordered, not adjacent, first occurrences kept
    edge_key = np.sort(eu * n + ev)
    chosen = np.zeros(0, dtype=np.int64)
    while len(chosen) < h:
        want = h - len(chosen)
        a = rng.integers(0, n, size=2 * want + 64)
        b = rng.integers(0, n, size=2 * want + 64)
        ok = a != b
        key = np.minimum(a, b)[ok] * n + np.maximum(a, b)[ok]
        pos = np.searchsorted(edge_key, key)
        adj = (pos < m) & (edge_key[np.minimum(pos, max(m - 1, 0))] == key) if m > 0 else np.zeros(len(key), dtype=bool)
        key = np.concatenate([chosen, key[~adj]])
        _, first = np.unique(key, return_index=True)
        chosen = key[np.sort(first)][:h]
    ne_u, ne_v = chosen // n, chosen % n
    # training lists: every directed entry whose pair was not held out, in the original order
    dkey = np.minimum(u, v) * n + np.maximum(u, v)
    pos = np.searchsorted(ho_e_key, dkey)
    held = (pos < h) & (ho_e_key[np.minimum(pos, max(h - 1, 0))] == dkey) if h > 0 else np.zeros(len(dkey), dtype=bool)
    tr_rowptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(u[~held], minlength=n), out=tr_rowptr[1:])
    tr_col = np.ascontiguousarray(col[~held])
    # held-out lists: both directions, labelled
    he_u, he_v = ho_e_key // n, ho_e_key % n
    a = np.concatenate([he_u, he_v, ne_u, ne_v])
    b = np.concatenate([he_v, he_u, ne_v, ne_u])
    lab = np.concatenate([np.ones(2 * h, dtype=np.uint8), np.zeros(2 * h, dtype=np.uint8)])
    ho_rowptr, ho_col, ho_is_edge = _csr(n, a, b, lab)
    return Split(tr_rowptr, tr_col, ho_rowptr, ho_col, np.ascontiguousarray(ho_is_edge))
