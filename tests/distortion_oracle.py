"""numpy / scipy oracle of the graph-reconstruction distortion (sympa_b200.metrics): hop distances by scipy's
csgraph, the per-row terms of sympa_distortion_rows and the two distortion figures over (pair, distance) lists -
the reference's route, which scores the scaled distances of its triplets."""
import numpy as np
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import shortest_path


def hop_matrix(ptr, idx, rows=None):
    """(R, N) int32 hop distances from the sources `rows` (default all nodes) of the undirected CSR graph,
    -1 where a node is unreachable"""
    ptr, idx = np.asarray(ptr), np.asarray(idx)
    n = ptr.size - 1
    a = csr_matrix((np.ones(idx.size), idx, ptr), shape=(n, n))
    d = shortest_path(a, directed=False, unweighted=True, indices=rows)
    d = np.atleast_2d(d)
    out = np.full(d.shape, -1, dtype=np.int32)
    ok = np.isfinite(d)
    out[ok] = d[ok].astype(np.int32)
    return out


def distortion_rows(dist_block, hop_block, row_begin, scale):
    """per row u of the block, over the columns w > u with hop distance >= 1: (sum of |s d - g| / g, count,
    max of s d / g, min of s d / g); NaN in the three float terms when a scaled distance is NaN, -inf / +inf
    extremes for a row without pairs"""
    rows = dist_block.shape[0]
    out = (np.zeros(rows), np.zeros(rows, dtype=np.int64), np.full(rows, -np.inf), np.full(rows, np.inf))
    for r in range(rows):
        u = row_begin + r
        g = hop_block[r, u + 1:]
        keep = g >= 1
        sd = scale * dist_block[r, u + 1:][keep]
        g = g[keep].astype(np.float64)
        out[1][r] = sd.size
        if sd.size == 0:
            continue
        if np.isnan(sd).any():
            out[0][r] = out[2][r] = out[3][r] = np.nan
            continue
        out[0][r] = np.sum(np.abs(sd - g) / g)
        out[2][r] = np.max(sd / g)
        out[3][r] = np.min(sd / g)
    return out


def distortion(scaled_dist, graph_dist):
    """(average, worst-case) distortion over pairs: the scaled manifold distances and their hop distances"""
    sd = np.asarray(scaled_dist, dtype=np.float64)
    g = np.asarray(graph_dist, dtype=np.float64)
    ratio = sd / g
    return float(np.mean(np.abs(sd - g) / g)), float(np.max(ratio) / np.min(ratio))
