"""The definition of filtered link-prediction ranks (sympa_target_ranks, metrics.link_prediction) in numpy, by brute
force per pair: with d row u of the distance matrix and F(u) the filter row of u,

    C(u, v)  = {w in [0, N) : w != u, w != v, w not in F(u)}
    lt       = |{w in C : d(u,w) <  d(u,v)}|,    le = |{w in C : d(u,w) <= d(u,v)}|

-0.0 equals +0.0 (numpy's comparisons already say so); a NaN anywhere in row u (w != u) gives lt = le = -1."""
import numpy as np


def counts(row, u, v, filt):
    """(lt, le) of the pair (u, v) on the distance row `row` of u, filt the filter row of u (any iterable of ids)"""
    row = np.asarray(row, dtype=np.float64)
    others = np.arange(row.size) != u
    if np.isnan(row[others]).any():
        return -1, -1
    keep = others & (np.arange(row.size) != v)
    for w in filt:
        if 0 <= w < row.size:
            keep[w] = False
    comp = row[keep]
    x = row[v]
    return int((comp < x).sum()), int((comp <= x).sum())


def ranks(lt, le):
    """(rank, optimistic, pessimistic) as float64 arrays, NaN where lt < 0"""
    lt = np.asarray(lt, dtype=np.float64)
    le = np.asarray(le, dtype=np.float64)
    bad = lt < 0
    out = (1.0 + 0.5 * (lt + le), 1.0 + lt, 1.0 + le)
    return tuple(np.where(bad, np.nan, r) for r in out)


def pair_counts(dist_matrix, pairs, ptr, idx):
    """(lt, le) int64 arrays of every pair (u, v) of `pairs` on the full matrix, the filter the CSR (ptr, idx)"""
    d = np.asarray(dist_matrix)
    ptr, idx = np.asarray(ptr), np.asarray(idx)
    lt = np.empty(len(pairs), dtype=np.int64)
    le = np.empty(len(pairs), dtype=np.int64)
    for i, (u, v) in enumerate(np.asarray(pairs).tolist()):
        lt[i], le[i] = counts(d[u], u, v, idx[ptr[u]:ptr[u + 1]].tolist())
    return lt, le
