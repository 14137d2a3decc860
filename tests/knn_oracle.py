"""The definition of exact k-nearest-neighbour selection (sympa_row_topk, metrics.nearest) in numpy: row r of the
result is the stable ascending sort of the row with column exclude[r] removed (-0.0 and +0.0 compare equal, so they
keep their column order), cut to k, with every NaN entry and every missing entry replaced by (-1, NaN)."""
import numpy as np


def topk(block, k, exclude=None):
    """(ids (R, k) int64, values (R, k) float64) of the (R, M) array `block`; exclude: R columns, -1 for none"""
    block = np.asarray(block, dtype=np.float64)
    rows, cols = block.shape
    ids = np.full((rows, k), -1, dtype=np.int64)
    vals = np.full((rows, k), np.nan)
    for r in range(rows):
        keep = np.arange(cols)
        if exclude is not None:
            keep = keep[keep != exclude[r]]
        row = block[r, keep]
        order = np.argsort(row, kind="stable")[:k]          # NaN sorts last
        sel_ids, sel_vals = keep[order], row[order]
        sel_ids[np.isnan(sel_vals)] = -1
        ids[r, : order.size] = sel_ids
        vals[r, : order.size] = sel_vals
    return ids, vals
