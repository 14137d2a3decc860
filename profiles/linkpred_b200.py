"""Link-prediction evaluation on the GPU (sympa_b200.metrics.link_prediction: sympa_dist_rows, then
sympa_target_ranks, per block of distinct query rows): time of the whole call, time of the rank kernel alone on the
same block shapes (CUDA events) with its share of the call and its read rate, peak device memory, and the ranks
against a brute-force oracle on the device.

    python profiles/linkpred_b200.py [--out profiles/linkpred_b200.json] [--quick]

Workloads (held-out edges split by graphs.split_edges, seed 0, ranked in both directions, filter = the whole graph;
upper_spread tables, seed 0):
- config 3 (product_cartesian_triplets(3, 3, 5, 3): 5000 nodes, upper finf n = 6), 10 % held out;
- the random recursive tree of 2^17 nodes of eval_b200.py (the parent of k drawn from [0, k)), 5 % held out, at
  upper riem n = 4 and n = 2 (where the distances are cheapest and the rank kernel's share the largest);
- the random recursive tree of 2^20 nodes, 4096 held-out edges, at upper riem n = 4.
Each workload is warmed up by one untimed call; the call's time ends in the status check's synchronise.  Blocks of
1 GB of distances, larger than L2 (config 3's 5000-node rows fit 26 843 to a block: its call is one block of 8 bytes
x 5000 per distinct query node).  The kernel-alone time runs sympa_target_ranks on a block of uniform random distances
of the full block height with the targets of the first block's query nodes, scaled to the number of blocks; it reads
8 bytes per entry of the block.  The oracle: the matrix row of the query (dist_matrix, one call per query node),
then per pair the competitors counted on the device; every pair at 5000 nodes, the pairs of the first 64 query
nodes elsewhere.
Sanity leg on config 3, reported and not asserted: MRR and Hits@10 of the held-out edges before training and after 5
epochs of FusedEpochRunner (batch 131 072, lr 1e-2) on pairs PairSampler draws from the training graph."""
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


def setup(n_nodes, n, metric):
    import siegel_oracle as so
    from sympa_b200 import MetricType, UpperHalfManifold

    dev = torch.device("cuda", 0)
    table = so.upper_spread(n_nodes, n, generator=torch.Generator().manual_seed(0), scale=0.3).to(dev)
    man = UpperHalfManifold(dims=n, metric=MetricType.from_str(metric)).to(dev)
    return man, table


def grouped(pairs):
    """(distinct query nodes, target ptr, target idx) as link_prediction groups them"""
    order = torch.sort(pairs[:, 0], stable=True).indices
    nodes, counts = torch.unique_consecutive(pairs[order, 0], return_counts=True)
    ptr = torch.zeros(nodes.numel() + 1, dtype=torch.int64, device=pairs.device)
    torch.cumsum(counts, 0, out=ptr[1:])
    return nodes, ptr, pairs[order, 1].contiguous()


def oracle_mismatches(man, table, pairs, res, filt, max_nodes):
    """pairs of the first max_nodes distinct query nodes whose three ranks differ from the brute-force count"""
    ptr, idx = filt
    nodes = torch.unique(pairs[:, 0])[:max_nodes]
    n_nodes = table.shape[0]
    rank = torch.full((pairs.shape[0],), float("nan"), dtype=torch.float64, device=pairs.device)
    rank[res.pairs] = res.rank
    opt = torch.full_like(rank, float("nan"))
    opt[res.pairs] = res.optimistic
    bad = checked = 0
    for u in nodes.tolist():
        row = man.dist_matrix(table, u, 1)[0]
        keep = torch.ones(n_nodes, dtype=torch.bool, device=row.device)
        keep[u] = False
        keep[idx[ptr[u]:ptr[u + 1]]] = False
        for i in (pairs[:, 0] == u).nonzero()[:, 0].tolist():
            v = int(pairs[i, 1])
            k = keep.clone()
            k[v] = False
            comp = row[k]
            lt, le = int((comp < row[v]).sum()), int((comp <= row[v]).sum())
            bad += not (rank[i].item() == 1 + (lt + le) / 2 and opt[i].item() == 1 + lt)
            checked += 1
    return checked, bad


def kernel_time(n_nodes, nodes, t_ptr, t_idx, filt, block, reps=5):
    """target_ranks alone on a (block, N) block of uniform distances in [0, 10) with the first block's targets"""
    from sympa_b200 import ops

    rows = min(block, nodes.numel())
    d = torch.rand(rows, n_nodes, dtype=torch.float64, device="cuda") * 10
    q = nodes[:rows]
    out = (torch.empty_like(t_idx), torch.empty_like(t_idx))
    ops.target_ranks(d, q, (t_ptr[:rows + 1], t_idx), filt, out=out)
    t, _ = timed(lambda: ops.target_ranks(d, q, (t_ptr[:rows + 1], t_idx), filt, out=out), reps=reps)
    del d
    ops.check_status()
    return t * nodes.numel() / rows, 8 * rows * n_nodes / t


def workload(name, n_nodes, edges, n, metric, fraction, block_bytes, oracle_nodes):
    from sympa_b200 import graphs
    from sympa_b200.metrics import link_prediction

    dev = torch.device("cuda", 0)
    man, table = setup(n_nodes, n, metric)
    _, test = graphs.split_edges(edges, n_nodes, fraction)
    pairs = torch.cat((test, test.flip(1))).to(dev)
    filt = graphs.adjacency_csr(edges.to(dev), n_nodes)
    link_prediction(man, table, pairs, filt, block_bytes=block_bytes)             # warm-up
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    t, res = timed(lambda: link_prediction(man, table, pairs, filt, block_bytes=block_bytes))
    peak = torch.cuda.max_memory_allocated() - base
    nodes, t_ptr, t_idx = grouped(pairs)
    block = max(1, min(block_bytes // (8 * n_nodes), nodes.numel()))
    blocks = -(-nodes.numel() // block)
    t_kernel, read_rate = kernel_time(n_nodes, nodes, t_ptr, t_idx, filt, block)
    checked, bad = oracle_mismatches(man, table, pairs, res, filt, oracle_nodes)
    rec = {"workload": name, "nodes": n_nodes, "edges": int(edges.shape[0]), "kind": "upper", "n": n, "metric": metric,
           "held_out_edges": int(test.shape[0]), "pairs": int(pairs.shape[0]), "query_nodes": int(nodes.numel()),
           "block_rows": block, "blocks": blocks, "mrr": res.mrr, "hits": res.hits,
           "call_sec": t, "distances_per_sec": nodes.numel() * n_nodes / t,
           "target_ranks_sec_est": t_kernel, "target_ranks_share_est": t_kernel / t,
           "target_ranks_read_gb_per_sec": read_rate / 1e9,
           "peak_device_bytes_over_inputs": int(peak),
           "oracle_pairs_checked": checked, "oracle_mismatched_pairs": bad}
    print(json.dumps(rec), flush=True)
    del man, table
    torch.cuda.empty_cache()
    return rec


def sanity(cfg3, epochs):
    from sample_b200 import model_for
    from sympa_b200 import graphs
    from sympa_b200.runner import FusedEpochRunner
    from sympa_b200.sampling import PairSampler

    dev = torch.device("cuda", 0)
    ids, gd, n_nodes = graphs.product_cartesian_triplets(*cfg3)
    edges = ids[gd == 1]
    train, test = graphs.split_edges(edges, n_nodes, 0.1)
    pairs = torch.cat((test, test.flip(1))).to(dev)
    filt = graphs.adjacency_csr(edges.to(dev), n_nodes)
    adj = graphs.adjacency_csr(train.to(dev), n_nodes)
    sources = int((adj[0][1:] > adj[0][:-1]).sum())
    per_source = -(-ids.shape[0] // n_nodes)
    model = model_for(n_nodes, "upper", 6, "finf", dev)
    before = model.link_prediction(pairs, filt)
    sampler = PairSampler(adj, sources, per_source, seed=0)
    s_ids, s_gd = sampler.sample(0)
    runner = FusedEpochRunner(model, 1e-2, s_ids, s_gd, 131072, device_shuffle=True)
    for e in range(epochs):
        sampler.sample(e, out=(runner.ids, runner.gdist))
        runner.run_epoch(e)
    after = model.link_prediction(pairs, filt)
    rec = {"graph": "config3_product_cartesian", "nodes": n_nodes, "edges": int(edges.shape[0]),
           "train_edges": int(train.shape[0]), "held_out_edges": int(test.shape[0]), "pairs": int(pairs.shape[0]),
           "kind": "upper", "n": 6, "metric": "finf", "epochs": epochs, "batch": 131072, "lr": 1e-2,
           "sampled_sources": sources, "sampled_pairs_per_source": per_source,
           "mrr_before": before.mrr, "hits10_before": before.hits[10],
           "mrr_after": after.mrr, "hits10_after": after.hits[10]}
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small sizes (a check of the script, not a measurement)")
    ap.add_argument("--block-bytes", type=int, default=1 << 30)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "linkpred_b200.py measures on the GPU"
    from sympa_b200 import graphs

    torch.cuda.set_device(0)
    if a.quick:
        cfg3, mid, big, big_held, epochs = (2, 2, 3, 2), 1 << 11, 1 << 12, 256, 1
    else:
        cfg3, mid, big, big_held, epochs = (3, 3, 5, 3), 1 << 17, 1 << 20, 4096, 5
    ids, gd, n3 = graphs.product_cartesian_triplets(*cfg3)
    records = [workload("config3_product_cartesian", n3, ids[gd == 1], 6, "finf", 0.1, a.block_bytes, n3)]
    del ids, gd
    tree = random_tree(mid)
    for n in (4, 2):
        records.append(workload(f"random_tree_{mid}", mid, tree, n, "riem", 0.05, a.block_bytes, 64))
    tree = random_tree(big)
    records.append(workload(f"random_tree_{big}", big, tree, 4, "riem", big_held / (big - 1), a.block_bytes, 64))
    quality = sanity(cfg3, epochs)
    out = {"gpu": gpu_info(), "torch": torch.__version__, "block_bytes": a.block_bytes, "quick": a.quick,
           "records": records, "sanity_config3": quality}
    text = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print("wrote", a.out)


if __name__ == "__main__":
    main()
