"""Graph-reconstruction evaluation on the GPU (sympa_b200.metrics.evaluate: distortion and mAP in one pass over row
blocks of the distance matrix): time of the whole evaluation, time of the same dist_matrix blocks alone, the hop
(breadth-first search), distortion and AP kernels per full block and their shares, peak device memory, and - for
BASELINE config 3 - the host route (scipy csgraph hop distances, then the numpy formula over the triplets on the
distances of dist_from_table).

    python profiles/eval_b200.py [--out profiles/eval_b200.json] [--quick]

Workloads, those of map_eval.py: config 3 (product_cartesian_triplets(3, 3, 5, 3): 5000 nodes, upper finf n = 6),
a balanced tree of branching 4 and height 8 (87 381 nodes, upper riem n = 4) and a random recursive tree of 2^17
nodes (the parent of k drawn from [0, k), upper riem n = 2).  Times are CUDA events after one untimed warm-up
evaluation; the blocks (1 GB of distances + hop distances each) are larger than L2 except config 3's (300 MB in
one block)."""
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
sys.path.insert(0, os.path.join(ROOT, "tests"))


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


def timed(fn, reps=1):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for _ in range(reps):
        out = fn()
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / 1e3 / reps, out


def workload(name, n_nodes, edges, kind, n, metric, block_bytes, host_route):
    import siegel_oracle as so
    from sympa_b200 import MetricType, UpperHalfManifold, graphs, ops
    from sympa_b200.metrics import evaluate

    dev = torch.device("cuda", 0)
    scale = 1.0
    adj = graphs.adjacency_csr(edges, n_nodes)
    adj_dev = (adj[0].to(dev), adj[1].to(dev))
    table = so.upper_spread(n_nodes, n, generator=torch.Generator().manual_seed(0), scale=0.3).to(dev)
    man = UpperHalfManifold(dims=n, metric=MetricType.from_str(metric)).to(dev)
    evaluate(man, table, adj_dev, scale=scale, block_bytes=block_bytes)          # warm-up: every shape below
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    t_eval, r = timed(lambda: evaluate(man, table, adj_dev, scale=scale, block_bytes=block_bytes))
    peak = torch.cuda.max_memory_allocated() - base

    block = max(1, min(block_bytes // (12 * n_nodes), n_nodes))
    buf = torch.empty(block, n_nodes, dtype=torch.float64, device=dev)
    hop = torch.empty(block, n_nodes, dtype=torch.int32, device=dev)

    def dist_only():
        for r0 in range(0, n_nodes, block):
            rc = min(block, n_nodes - r0)
            ops.dist_matrix(kind, metric, table, r0, rc, out=buf[:rc])
    dist_only()
    t_dist, _ = timed(dist_only)
    # each kernel alone on one full block (rows [0, block)), scaled to the number of blocks
    reps = 3
    ap_out = torch.empty(block, dtype=torch.float64, device=dev)
    dr_out = ops.DistortionRows(*(torch.empty(block, dtype=t, device=dev)
                                  for t in (torch.float64, torch.int64, torch.float64, torch.float64)))
    ops.hop_distances(adj_dev, 0, block, out=hop)
    t_hop, _ = timed(lambda: ops.hop_distances(adj_dev, 0, block, out=hop), reps=reps)
    ops.distortion_rows(buf, hop, 0, scale, out=dr_out)
    t_dst, _ = timed(lambda: ops.distortion_rows(buf, hop, 0, scale, out=dr_out), reps=reps)
    ops.average_precision(buf, 0, adj_dev, out=ap_out)
    t_ap, _ = timed(lambda: ops.average_precision(buf, 0, adj_dev, out=ap_out), reps=reps)
    blocks = -(-n_nodes // block)
    ops.check_status()
    pairs = n_nodes * n_nodes
    entries = int(adj[1].numel())
    # entries of the first block's upper part, the distortion kernel's 12 bytes each
    upper = sum(n_nodes - 1 - u for u in range(block))
    rec = {"workload": name, "nodes": n_nodes, "adj_entries": entries, "kind": kind, "n": n, "metric": metric,
           "block_rows": block, "blocks": blocks, "scale": scale,
           "average_distortion": r.average_distortion, "worst_case_distortion": r.worst_case_distortion, "map": r.mean_ap,
           "eval_sec": t_eval, "eval_pairs_per_sec": pairs / t_eval,
           "dist_matrix_sec": t_dist, "dist_matrix_pairs_per_sec": pairs / t_dist,
           "metrics_share_by_difference": (t_eval - t_dist) / t_eval,
           "hop_kernel_sec_per_block": t_hop, "hop_kernel_sec_est_total": t_hop * blocks,
           "hop_kernel_share_est": t_hop * blocks / t_eval,
           "hop_kernel_visits_per_sec": block * (n_nodes + entries) / t_hop,
           "distortion_kernel_sec_per_block": t_dst, "distortion_kernel_sec_est_total": t_dst * blocks,
           "distortion_kernel_share_est": t_dst * blocks / t_eval,
           "distortion_kernel_bytes_per_sec_first_block": 12 * upper / t_dst,
           "ap_kernel_sec_per_block": t_ap, "ap_kernel_share_est": t_ap * blocks / t_eval,
           "peak_device_bytes_over_inputs": int(peak), "full_matrix_bytes": 8 * pairs,
           "full_hop_matrix_bytes": 4 * pairs}
    if host_route:
        from distortion_oracle import distortion
        from scipy.sparse import csr_matrix
        from scipy.sparse.csgraph import shortest_path
        ptr, idx = adj[0].numpy(), adj[1].numpy()
        t0 = time.perf_counter()
        g = shortest_path(csr_matrix((np.ones(idx.size), idx, ptr), shape=(n_nodes, n_nodes)), directed=False,
                          unweighted=True)
        iu, ju = np.triu_indices(n_nodes, 1)
        gd = g[iu, ju]
        ok = np.isfinite(gd)
        iu, ju, gd = iu[ok], ju[ok], gd[ok]
        rec["host_scipy_hop_distances_sec"] = time.perf_counter() - t0
        ids = torch.from_numpy(np.stack((iu, ju), 1)).to(dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.no_grad():
            sd = (man.dist_from_table(table, ids) * scale).cpu().numpy()
        rec["host_route_dist_from_table_sec"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        avg, worst = distortion(sd, gd)
        rec["host_numpy_formula_sec"] = time.perf_counter() - t0
        rec["host_average_distortion"], rec["host_worst_case_distortion"] = avg, worst
        rec["host_vs_device_average_rel_diff"] = abs(r.average_distortion - avg) / abs(avg)
        rec["host_vs_device_worst_case_rel_diff"] = abs(r.worst_case_distortion - worst) / abs(worst)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small sizes (a check of the script, not a measurement)")
    ap.add_argument("--block-bytes", type=int, default=1 << 30)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "eval_b200.py measures on the GPU"
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
