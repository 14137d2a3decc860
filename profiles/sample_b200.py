"""Training pairs sampled on the GPU (sympa_b200.sampling.PairSampler, sympa_sample_pairs): what sampling costs, how
it compares with the training epoch it feeds, and what training from sampled pairs gives against all triplets.

    python profiles/sample_b200.py [--out profiles/sample_b200.json] [--quick]

1. sampler: time per call, sources/s, breadth-first-search visits/s ((N + adjacency entries) per source, what one
   search touches) and pairs/s, at K = 64 and 1024 pairs per source, for config 3 (product_cartesian_triplets(3, 3,
   5, 3): 5000 nodes), the balanced 4-ary tree of height 8 (87 381 nodes) and a random recursive tree of 2^20 nodes
   (the parent of k drawn from [0, k); its visited set is in global memory).  CUDA events over 3 calls after one
   untimed call.
2. one sampled epoch on the 2^20-node tree, split into the sampler call and FusedEpochRunner.run_epoch (pairs written
   in place, the epoch replayed from its CUDA graph), for upper riem n = 4 and upper finf n = 6, batch 131 072, at
   several K with the sources per epoch fixed: where the search stops bounding the epoch.
3. config 3 (upper finf n = 6, batch 131 072, lr 1e-2 - bench.py's config): Model.evaluate (average distortion, mAP)
   after the same number of FusedEpochRunner epochs trained from all 12 497 500 triplets and from sampled pairs, 5000
   sources x 2500 pairs = 12 500 000 pairs per epoch."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from eval_b200 import gpu_info, timed  # noqa: E402


def random_tree_edges(n, seed=0):
    rng = np.random.default_rng(seed)
    k = torch.arange(1, n)
    parent = torch.from_numpy((rng.random(n - 1) * np.arange(1, n)).astype(np.int64))
    return torch.stack((k, parent), 1)


def sampler_record(name, adj, sources, k):
    from sympa_b200 import ops
    from sympa_b200.sampling import PairSampler
    sampler = PairSampler(adj, sources, k, seed=1)
    src = sampler.epoch_sources(0)
    ids, gd = sampler.sample(0)
    reps = 3
    t, _ = timed(lambda: ops.sample_pairs(sampler.adj, src, k, 1, 0, out=(ids, gd)), reps=reps)
    ops.check_status()
    n_nodes, entries = adj[0].numel() - 1, adj[1].numel()
    return {"graph": name, "nodes": n_nodes, "adj_entries": entries, "sources": sources, "pairs_per_source": k,
            "pairs": sources * k, "sample_sec": t, "sources_per_sec": sources / t,
            "bfs_visits_per_sec": sources * (n_nodes + entries) / t, "pairs_per_sec": sources * k / t,
            "workspace_bytes": int(ops._sample_workspace[("cuda", torch.cuda.current_device())].numel() * 8),
            "mean_graph_distance": float(gd.mean())}


def model_for(n_nodes, kind, n, metric, dev):
    from types import SimpleNamespace
    from sympa_b200.model import Model
    torch.manual_seed(0)
    args = SimpleNamespace(manifold=kind, metric=metric, dims=n, num_points=n_nodes, scale_init=1.0, scale_coef=1.0,
                           train_scale=False)
    return Model(args).to(dev)


def epoch_record(adj, n_nodes, kind, n, metric, sources, k, batch, dev, epochs=3):
    from sympa_b200.runner import FusedEpochRunner
    from sympa_b200.sampling import PairSampler
    sampler = PairSampler(adj, sources, k, seed=2)
    model = model_for(n_nodes, kind, n, metric, dev)
    ids, gd = sampler.sample(0)
    runner = FusedEpochRunner(model, 1e-2, ids, gd, batch, device_shuffle=True)
    runner.run_epoch(0)                                  # capture and warm-up
    t_sample = t_train = 0.0
    for e in range(1, epochs + 1):
        ts, _ = timed(lambda: sampler.sample(e, out=(runner.ids, runner.gdist)))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss = runner.run_epoch(e)                       # reads the loss back: ends synchronised
        t_train += time.perf_counter() - t0
        t_sample += ts
    t_sample, t_train = t_sample / epochs, t_train / epochs
    return {"graph_nodes": n_nodes, "kind": kind, "n": n, "metric": metric, "sources": sources, "pairs_per_source": k,
            "pairs_per_epoch": sources * k, "batch": batch, "steps": runner.steps, "sample_sec": t_sample,
            "run_epoch_sec": t_train, "sample_share": t_sample / (t_sample + t_train),
            "epoch_pairs_per_sec": sources * k / (t_sample + t_train), "last_loss": loss}


def quality_record(epochs, dev, cfg3):
    from sympa_b200 import graphs
    from sympa_b200.runner import FusedEpochRunner
    from sympa_b200.sampling import PairSampler
    ids, gd, n_nodes = graphs.product_cartesian_triplets(*cfg3)
    adj = graphs.adjacency_csr(ids[gd == 1], n_nodes)
    adj = (adj[0].to(dev), adj[1].to(dev))
    ids, gd = ids.to(dev), gd.to(dev)
    per_source = -(-ids.shape[0] // n_nodes)
    rec = {"graph": "config3_product_cartesian", "nodes": n_nodes, "triplets": ids.shape[0], "epochs": epochs,
           "kind": "upper", "n": 6, "metric": "finf", "batch": 131072, "lr": 1e-2,
           "sampled_sources": n_nodes, "sampled_pairs_per_source": per_source, "sampled_pairs_per_epoch": n_nodes * per_source}
    model = model_for(n_nodes, "upper", 6, "finf", dev)
    rec["initial_average_distortion"], rec["initial_map"] = model.evaluate(adj)
    runner = FusedEpochRunner(model, 1e-2, ids, gd, 131072, device_shuffle=True)
    for e in range(epochs):
        runner.run_epoch(e)
    rec["triplets_average_distortion"], rec["triplets_map"] = model.evaluate(adj)
    del runner, ids, gd
    model = model_for(n_nodes, "upper", 6, "finf", dev)
    sampler = PairSampler(adj, n_nodes, per_source, seed=0)
    s_ids, s_gd = sampler.sample(0)
    runner = FusedEpochRunner(model, 1e-2, s_ids, s_gd, 131072, device_shuffle=True)
    for e in range(epochs):
        sampler.sample(e, out=(runner.ids, runner.gdist))
        runner.run_epoch(e)
    rec["sampled_average_distortion"], rec["sampled_map"] = model.evaluate(adj)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small sizes (a check of the script, not a measurement)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "sample_b200.py measures on the GPU"
    from sympa_b200 import graphs

    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    if a.quick:
        cfg3, (tb, th), rnd, big_sources, epochs, ks = (2, 2, 3, 2), (2, 3), 1 << 12, 64, 1, (16, 64)
    else:
        cfg3, (tb, th), rnd, big_sources, epochs, ks = (3, 3, 5, 3), (4, 8), 1 << 20, 4096, 5, (64, 256, 1024, 4096)
    ids, gd, n3 = graphs.product_cartesian_triplets(*cfg3)
    graphs_ = [("config3_product_cartesian", graphs.adjacency_csr(ids[gd == 1], n3), min(n3, 5000))]
    del ids, gd
    nt = (tb ** (th + 1) - 1) // (tb - 1)
    k = torch.arange(1, nt)
    graphs_.append((f"balanced_tree_{tb}_{th}", graphs.adjacency_csr(torch.stack((k, (k - 1) // tb), 1), nt), min(nt, 8192)))
    tree = graphs.adjacency_csr(random_tree_edges(rnd), rnd)
    graphs_.append((f"random_tree_{rnd}", tree, big_sources))
    sampling = []
    for name, adj, sources in graphs_:
        adj = (adj[0].to(dev), adj[1].to(dev))
        for kk in (64, 1024):
            sampling.append(sampler_record(name, adj, sources, kk))
            print(json.dumps(sampling[-1]), flush=True)
    tree = (tree[0].to(dev), tree[1].to(dev))
    epochs_ = []
    for n, metric in ((4, "riem"), (6, "finf")):
        for kk in ks:
            epochs_.append(epoch_record(tree, rnd, "upper", n, metric, big_sources, kk, 131072, dev))
            print(json.dumps(epochs_[-1]), flush=True)
    quality = quality_record(epochs, dev, cfg3)
    print(json.dumps(quality), flush=True)
    out = {"gpu": gpu_info(), "torch": torch.__version__, "quick": a.quick, "sampling": sampling, "sampled_epoch": epochs_,
           "quality_config3": quality}
    text = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
