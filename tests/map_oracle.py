"""numpy oracle of the graph-reconstruction average precision (sympa_b200.metrics): the closed form of the
definition and the argsort-and-scan loop it restates.  Both take one row of distances, the row's node u and its
neighbour list; NaN for a node without neighbours."""
import numpy as np


def ap_closed_form(row, u, nbrs):
    """1/|N| sum_{v in N} |{v' in N : d_v' <= d_v}| / |{w != u : d_w <= d_v}|"""
    nbrs = np.asarray(nbrs, dtype=np.int64)
    if nbrs.size == 0:
        return float("nan")
    row = np.asarray(row, dtype=np.float64)
    others = np.sort(np.delete(row, u))
    dn = row[nbrs]
    hits = np.searchsorted(np.sort(dn), dn, side="right")      # |{v' in N : d_v' <= d_v}|
    ranks = np.searchsorted(others, dn, side="right")          # |{w != u : d_w <= d_v}|
    return float(np.mean(hits / ranks))


def ap_argsort_loop(row, u, nbrs):
    """sort the row, skip the node itself, record hits / i at the i-th hit (tie-free rows only)"""
    nbrs = set(int(v) for v in nbrs)
    if not nbrs:
        return float("nan")
    order = np.argsort(row, kind="stable")
    hits, i, acc = 0, 0, 0.0
    for w in order:
        if w == u:
            continue
        i += 1
        if int(w) in nbrs:
            hits += 1
            acc += hits / i
    return acc / len(nbrs)


def ap_rows(block, row_begin, ptr, idx, fn=ap_closed_form):
    """per-row AP of the (R, N) block holding rows [row_begin, row_begin + R)"""
    ptr, idx = np.asarray(ptr), np.asarray(idx)
    return np.array([fn(block[r], row_begin + r, idx[ptr[row_begin + r]: ptr[row_begin + r + 1]])
                     for r in range(block.shape[0])])
