"""Exact k-nearest-neighbour queries on the GPU (sympa_b200.metrics.nearest: sympa_dist_rows, then sympa_row_topk,
per block of query rows): time of the whole call, time of the selection kernel alone on the same block shapes (CUDA
events) with its share of the call and its read rate, and the outputs against the stable sort of the distance
matrix rows.

    python profiles/knn_b200.py [--out profiles/knn_b200.json] [--quick]

Workloads: the table sizes of eval_b200.py / estimate_b200.py, 2^17 and 2^20 nodes (upper_spread tables, seed 0,
the graph plays no part), at upper riem n = 4, upper finf n = 6 and upper riem n = 10 (2^20 nodes: Q = 1 and 1024
only, its distances cost the most), plus upper riem n = 2 at 2^17 nodes, where the distances are cheapest and the
selection's share the largest.  Q = 1, 1024 and 4096 random query ids, k = 10 and 1024.  Each (table, k) is warmed
up on one block first; times are CUDA events around one call, which ends in a device synchronise (the status check).
Blocks of 1 GB of distances (128 rows at 2^20 nodes, 1024 at 2^17), larger than L2; a single query row (8 MB at
2^20 nodes) is not, so the Q = 1 selection reads it from L2 in the kernel-alone timing.  The selection reads 8 bytes
per entry.  The oracle: rows of dist_matrix (one call per query), torch.sort(stable=True) on the device with the
query's own column set to +inf, cut to k; every query at 2^17 nodes, the first 64 at 2^20."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from eval_b200 import gpu_info, timed  # noqa: E402


def setup(n_nodes, n, metric):
    import siegel_oracle as so
    from sympa_b200 import MetricType, UpperHalfManifold

    dev = torch.device("cuda", 0)
    table = so.upper_spread(n_nodes, n, generator=torch.Generator().manual_seed(0), scale=0.3).to(dev)
    man = UpperHalfManifold(dims=n, metric=MetricType.from_str(metric)).to(dev)
    return man, table


def oracle_mismatches(man, table, queries, got, k):
    """rows of `got` that differ from the stable sort of the matrix row (ids, or distance bits)"""
    bad = 0
    for i, u in enumerate(queries.tolist()):
        row = man.dist_matrix(table, u, 1)[0]
        row[u] = float("inf")
        s = torch.sort(row, stable=True)
        same_ids = torch.equal(s.indices[:k], got.ids[i])
        same_vals = torch.equal(s.values[:k].view(torch.int64), got.distances[i].view(torch.int64))
        bad += not (same_ids and same_vals)
    return bad


def topk_time(n_nodes, rows, k, reps):
    """row_topk alone on a (rows, N) block of distances of the same magnitudes (uniform in [0, 10))"""
    from sympa_b200 import ops

    block = torch.rand(rows, n_nodes, dtype=torch.float64, device="cuda") * 10
    exclude = torch.arange(rows, dtype=torch.int64, device="cuda")
    out = ops.row_topk(block, k, exclude=exclude)
    t, _ = timed(lambda: ops.row_topk(block, k, exclude=exclude, out=out), reps=reps)
    del block
    return t


def workload(n_nodes, n, metric, q_sizes, ks, oracle_rows, block_bytes, seed):
    from sympa_b200 import ops
    from sympa_b200.metrics import nearest

    man, table = setup(n_nodes, n, metric)
    rng = np.random.default_rng(seed)
    block = max(1, block_bytes // (8 * n_nodes))
    out = []
    for k in ks:
        nearest(man, table, torch.arange(min(block, n_nodes), device="cuda"), k, block_bytes=block_bytes)   # warm-up
        for q in q_sizes:
            queries = torch.from_numpy(rng.integers(0, n_nodes, q)).cuda()
            t, got = timed(lambda: nearest(man, table, queries, k, block_bytes=block_bytes))
            # the selection alone on the block shapes of this call: full blocks and the rest
            full, rest = divmod(q, block)
            t_sel = 0.0
            if full:
                t_sel += full * topk_time(n_nodes, block, k, reps=5)
            if rest:
                t_sel += topk_time(n_nodes, rest, k, reps=5)
            checked = min(q, oracle_rows)
            bad = oracle_mismatches(man, table, queries[:checked], got, k)
            ops.check_status()
            rec = {"nodes": n_nodes, "kind": "upper", "n": n, "metric": metric, "queries": q, "k": k,
                   "block_rows": min(block, q), "nearest_sec": t, "pairs_per_sec": q * n_nodes / t,
                   "row_topk_sec_est": t_sel, "row_topk_share_est": t_sel / t,
                   "row_topk_read_gb_per_sec": 8 * q * n_nodes / t_sel / 1e9,
                   "oracle_rows_checked": checked, "oracle_mismatched_rows": bad}
            print(json.dumps(rec), flush=True)
            out.append(rec)
    del man, table
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small sizes (a check of the script, not a measurement)")
    ap.add_argument("--block-bytes", type=int, default=1 << 30)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "knn_b200.py measures on the GPU"
    torch.cuda.set_device(0)
    if a.quick:
        mid, big, qs, ks, big_oracle = 1 << 11, 1 << 12, (1, 64, 200), (10, 1024), 16
    else:
        mid, big, qs, ks, big_oracle = 1 << 17, 1 << 20, (1, 1024, 4096), (10, 1024), 64
    records = []
    records += workload(mid, 2, "riem", qs, ks, qs[-1], a.block_bytes, 1)
    for n, metric in ((4, "riem"), (6, "finf"), (10, "riem")):
        records += workload(mid, n, metric, qs, ks, qs[-1], a.block_bytes, n)
    for n, metric in ((4, "riem"), (6, "finf")):
        records += workload(big, n, metric, qs, ks, big_oracle, a.block_bytes, n)
    records += workload(big, 10, "riem", qs[:2], ks, big_oracle, a.block_bytes, 10)
    out = {"gpu": gpu_info(), "torch": torch.__version__, "block_bytes": a.block_bytes, "quick": a.quick,
           "records": records}
    text = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print("wrote", a.out)


if __name__ == "__main__":
    main()
