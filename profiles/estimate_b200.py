"""Sampled-row estimates on the GPU (sympa_b200.metrics.estimate): time of estimate at several sample sizes on a
graph too large to evaluate in full, and, on graphs that can be, estimate against evaluate on the same table.

    python profiles/estimate_b200.py [--out profiles/estimate_b200.json] [--quick]

Workloads:
- the random recursive tree of 2^20 nodes (the parent of k drawn from [0, k), as in eval_b200.py) with tables of
  upper riem n = 4, upper finf n = 6 and upper riem n = 10: estimate at S = 256, 1024 and 4096 (n = 10 at S = 256
  and 1024 only: its distances cost the most);
- the random tree of 2^17 nodes (upper riem n = 2) and BASELINE config 3 (product_cartesian_triplets(3, 3, 5, 3):
  5000 nodes, upper finf n = 6), the workloads of eval_b200.py: evaluate and estimate at S = 1024 on the same table,
  both times and |estimate - exact| / standard error for both metrics.
Every shape is run once untimed first; times are CUDA events around one call, which ends in a device synchronise
(the status check).  Blocks of 1 GB of distances + hop distances each, larger than L2."""
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


def random_tree(n_nodes, seed=0):
    rng = np.random.default_rng(seed)
    k = torch.arange(1, n_nodes)
    parent = torch.from_numpy((rng.random(n_nodes - 1) * np.arange(1, n_nodes)).astype(np.int64))
    return torch.stack((k, parent), 1)


def setup(n_nodes, edges, n, metric):
    import siegel_oracle as so
    from sympa_b200 import MetricType, UpperHalfManifold, graphs

    dev = torch.device("cuda", 0)
    ptr, idx = graphs.adjacency_csr(edges, n_nodes)
    adj = (ptr.to(dev), idx.to(dev))
    table = so.upper_spread(n_nodes, n, generator=torch.Generator().manual_seed(0), scale=0.3).to(dev)
    man = UpperHalfManifold(dims=n, metric=MetricType.from_str(metric)).to(dev)
    return man, table, adj


def record(e):
    return {"mean_ap": e.mean_ap, "mean_ap_se": e.mean_ap_se, "average_distortion": e.average_distortion,
            "average_distortion_se": e.average_distortion_se,
            "sampled_worst_case_distortion": e.sampled_worst_case_distortion}


def large(name, n_nodes, edges, n, metric, sizes, block_bytes):
    from sympa_b200.metrics import estimate

    man, table, adj = setup(n_nodes, edges, n, metric)
    out = []
    for s in sizes:
        estimate(man, table, adj, s, block_bytes=block_bytes)                  # warm-up of this shape
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        t, e = timed(lambda: estimate(man, table, adj, s, block_bytes=block_bytes))
        peak = torch.cuda.max_memory_allocated() - base
        pairs = s * n_nodes
        out.append({"workload": name, "nodes": n_nodes, "adj_entries": int(adj[1].numel()), "kind": "upper", "n": n,
                    "metric": metric, "sample_rows": s, "estimate_sec": t, "pairs": pairs, "pairs_per_sec": pairs / t,
                    "peak_device_bytes_over_inputs": int(peak), **record(e)})
        print(json.dumps(out[-1]), flush=True)
    del man, table, adj
    torch.cuda.empty_cache()
    return out


def against_exact(name, n_nodes, edges, n, metric, s, block_bytes):
    from sympa_b200.metrics import estimate, evaluate

    man, table, adj = setup(n_nodes, edges, n, metric)
    evaluate(man, table, adj, block_bytes=block_bytes)
    t_eval, exact = timed(lambda: evaluate(man, table, adj, block_bytes=block_bytes))
    estimate(man, table, adj, s, block_bytes=block_bytes)
    t_est, e = timed(lambda: estimate(man, table, adj, s, block_bytes=block_bytes))
    rec = {"workload": name, "nodes": n_nodes, "kind": "upper", "n": n, "metric": metric, "sample_rows": s,
           "evaluate_sec": t_eval, "estimate_sec": t_est, "speedup": t_eval / t_est,
           "exact_mean_ap": exact.mean_ap, "exact_average_distortion": exact.average_distortion,
           "exact_worst_case_distortion": exact.worst_case_distortion, **record(e),
           "mean_ap_error_in_se": abs(e.mean_ap - exact.mean_ap) / e.mean_ap_se,
           "average_distortion_error_in_se": abs(e.average_distortion - exact.average_distortion) / e.average_distortion_se,
           "sampled_over_exact_worst_case": e.sampled_worst_case_distortion / exact.worst_case_distortion}
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small sizes (a check of the script, not a measurement)")
    ap.add_argument("--block-bytes", type=int, default=1 << 30)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "estimate_b200.py measures on the GPU"
    from sympa_b200 import graphs

    torch.cuda.set_device(0)
    if a.quick:
        big, sizes, mid, cfg3, s_cmp = 1 << 12, (16, 64), 1 << 10, (2, 2, 3, 2), 64
    else:
        big, sizes, mid, cfg3, s_cmp = 1 << 20, (256, 1024, 4096), 1 << 17, (3, 3, 5, 3), 1024
    edges = random_tree(big)
    records = []
    records += large(f"random_tree_{big}", big, edges, 4, "riem", sizes, a.block_bytes)
    records += large(f"random_tree_{big}", big, edges, 6, "finf", sizes, a.block_bytes)
    records += large(f"random_tree_{big}", big, edges, 10, "riem", sizes[:2], a.block_bytes)
    comparisons = [against_exact(f"random_tree_{mid}", mid, random_tree(mid), 2, "riem", s_cmp, a.block_bytes)]
    ids, gd, n3 = graphs.product_cartesian_triplets(*cfg3)
    comparisons.append(against_exact("config3_product_cartesian", n3, ids[gd == 1], 6, "finf", s_cmp, a.block_bytes))
    out = {"gpu": gpu_info(), "torch": torch.__version__, "block_bytes": a.block_bytes, "quick": a.quick,
           "estimates": records, "against_evaluate": comparisons}
    text = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print("wrote", a.out)


if __name__ == "__main__":
    main()
