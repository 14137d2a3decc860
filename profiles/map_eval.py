"""Graph-reconstruction mAP evaluation on the GPU (sympa_b200.metrics.mean_average_precision): time of the whole
streamed evaluation, time of the same dist_matrix blocks alone, the AP kernel's share, peak device memory, and -
for BASELINE config 3 - the host numpy argsort loop on the same distances.

    python profiles/map_eval.py [--out profiles/map_eval_b200.json] [--quick]

Workloads: config 3 (product_cartesian_triplets(3, 3, 5, 3): 5000 nodes, upper finf n = 6), a balanced tree of
branching 4 and height 8 (87 381 nodes, upper riem n = 4) and a random recursive tree of 2^17 nodes (the parent of
k drawn from [0, k), upper riem n = 2).  Times are CUDA events after one untimed warm-up evaluation; the distance
blocks (1 GB each) are larger than L2 except config 3's (200 MB in one block)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in r.stdout.strip().split(",")]
        info.update(smi_name=name, power_limit=power)
    except Exception as e:  # noqa: BLE001
        info["power_limit"] = f"not read: {e}"
    return info


def host_argsort_map(dm, ptr, idx):
    """the usual host loop: sort each row, skip the node, precision at every hit"""
    n = dm.shape[0]
    ap = np.full(n, np.nan)
    mask = np.zeros(n, dtype=bool)
    for u in range(n):
        nb = idx[ptr[u]:ptr[u + 1]]
        if nb.size == 0:
            continue
        mask[nb] = True
        order = np.argsort(dm[u])
        order = order[order != u]
        hit = mask[order]
        hits = np.cumsum(hit)
        ap[u] = np.mean(hits[hit] / (np.flatnonzero(hit) + 1))
        mask[nb] = False
    return ap


def timed(fn, reps=1):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(reps):
        out = fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / 1e3 / reps, out


def workload(name, n_nodes, edges, kind, n, metric, block_bytes, host_loop):
    import siegel_oracle as so
    from sympa_b200 import MetricType, UpperHalfManifold, graphs, ops
    from sympa_b200.metrics import mean_average_precision

    dev = torch.device("cuda", 0)
    adj = graphs.adjacency_csr(edges, n_nodes)
    adj_dev = (adj[0].to(dev), adj[1].to(dev))
    table = so.upper_spread(n_nodes, n, generator=torch.Generator().manual_seed(0), scale=0.3).to(dev)
    man = UpperHalfManifold(dims=n, metric=MetricType.from_str(metric)).to(dev)
    mean_average_precision(man, table, adj_dev, block_bytes=block_bytes)        # warm-up: every shape below
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    t_eval, (s, c, ap) = timed(lambda: mean_average_precision(man, table, adj_dev, block_bytes=block_bytes))
    peak = torch.cuda.max_memory_allocated() - base

    block = max(1, min(block_bytes // (8 * n_nodes), n_nodes))
    buf = torch.empty(block, n_nodes, dtype=torch.float64, device=dev)

    def dist_only():
        for r0 in range(0, n_nodes, block):
            rc = min(block, n_nodes - r0)
            ops.dist_matrix(kind, metric, table, r0, rc, out=buf[:rc])
    dist_only()
    t_dist, _ = timed(dist_only)
    # the AP kernel alone on one full block (distances already in buf), scaled to the number of blocks
    ap_out = torch.empty(block, dtype=torch.float64, device=dev)
    ops.average_precision(buf, 0, adj_dev, out=ap_out)
    t_ap_block, _ = timed(lambda: ops.average_precision(buf, 0, adj_dev, out=ap_out), reps=5)
    blocks = -(-n_nodes // block)
    ops.check_status()
    pairs = n_nodes * n_nodes
    rec = {"workload": name, "nodes": n_nodes, "adj_entries": int(adj[1].numel()), "kind": kind, "n": n, "metric": metric,
           "block_rows": block, "blocks": blocks, "map": s / c,
           "eval_sec": t_eval, "eval_pairs_per_sec": pairs / t_eval,
           "dist_matrix_sec": t_dist, "dist_matrix_pairs_per_sec": pairs / t_dist,
           "ap_share_by_difference": (t_eval - t_dist) / t_eval,
           "ap_kernel_sec_per_block": t_ap_block, "ap_kernel_sec_est_total": t_ap_block * blocks,
           "ap_kernel_share_est": t_ap_block * blocks / t_eval,
           "ap_kernel_bytes_per_sec_full_block": block * n_nodes * 8 / t_ap_block,
           "peak_device_bytes_over_inputs": int(peak), "full_matrix_bytes": 8 * pairs}
    if host_loop:
        dm = ops.dist_matrix(kind, metric, table).cpu().numpy()
        ptr, idx = adj[0].numpy(), adj[1].numpy()
        t0 = time.perf_counter()
        host = host_argsort_map(dm, ptr, idx)
        rec["host_numpy_argsort_loop_sec"] = time.perf_counter() - t0
        rec["host_numpy_map"] = float(np.nanmean(host))
        dev_ap = ap.cpu().numpy()
        ok = ~np.isnan(host)
        rec["host_vs_device_max_rel_diff"] = float(np.max(np.abs(dev_ap[ok] - host[ok]) / np.abs(host[ok])))
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small sizes (a check of the script, not a measurement)")
    ap.add_argument("--block-bytes", type=int, default=1 << 30)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "map_eval.py measures on the GPU"
    from sympa_b200 import graphs

    torch.cuda.set_device(0)
    rng = np.random.default_rng(0)
    if a.quick:
        cfg3, (tb, th), rnd = (2, 2, 3, 2), (2, 3), 1 << 10
    else:
        cfg3, (tb, th), rnd = (3, 3, 5, 3), (4, 8), 1 << 17
    ids, gd, n3 = graphs.product_cartesian_triplets(*cfg3)
    records = [workload("config3_product_cartesian", n3, ids[gd == 1], "upper", 6, "finf", a.block_bytes, True)]
    nt = (tb ** (th + 1) - 1) // (tb - 1)
    k = torch.arange(1, nt)
    records.append(workload(f"balanced_tree_{tb}_{th}", nt, torch.stack((k, (k - 1) // tb), 1), "upper", 4, "riem",
                            a.block_bytes, False))
    k = torch.arange(1, rnd)
    parent = torch.from_numpy((rng.random(rnd - 1) * np.arange(1, rnd)).astype(np.int64))
    records.append(workload(f"random_tree_{rnd}", rnd, torch.stack((k, parent), 1), "upper", 2, "riem", a.block_bytes, False))
    out = {"gpu": gpu_info(), "torch": torch.__version__, "block_bytes": a.block_bytes, "quick": a.quick, "records": records}
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
