"""Multi-GPU (NCCL) check of link-prediction evaluation; run under torchrun on >= 2 GPUs, e.g.
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multigpu/check_nccl_linkpred.py
(not collected by pytest).  Every rank ranks the pairs of its distributed.row_shard part of the distinct query nodes;
the all-reduced MRR, Hits@k and count must equal the single-rank ones, and each rank's per-pair ranks must be the
single-rank ranks of the same pairs."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def main():
    import siegel_oracle as so
    from sympa_b200 import MetricType, UpperHalfManifold, graphs
    from sympa_b200 import distributed as sd
    from sympa_b200.metrics import link_prediction

    rank, world, local = sd.init_process_group()
    dev = torch.device("cuda", local)
    ids, gd, n_nodes = graphs.product_cartesian_triplets(2, 2, 4, 2)
    edges = ids[gd == 1]
    _, test = graphs.split_edges(edges, n_nodes, 0.2, seed=3)
    pairs = torch.cat((test, test.flip(1))).to(dev)
    filt = graphs.adjacency_csr(edges, n_nodes)
    table = so.upper_spread(n_nodes, 3, generator=torch.Generator().manual_seed(0), scale=0.3).to(dev)
    man = UpperHalfManifold(dims=3, metric=MetricType.from_str("fone")).to(dev)
    kw = dict(ks=(1, 3, 10), block_bytes=8 * n_nodes * 5)
    one = link_prediction(man, table, pairs, filt, **kw)
    r = link_prediction(man, table, pairs, filt, world_size=world, rank=rank, **kw)
    assert torch.equal(r.rank, one.rank[r.pairs])
    assert torch.equal(r.optimistic, one.optimistic[r.pairs]) and torch.equal(r.pessimistic, one.pessimistic[r.pairs])
    assert r.count == one.count == pairs.shape[0]
    assert abs(r.mrr - one.mrr) <= 1e-13 * one.mrr, (r.mrr, one.mrr)
    assert r.hits == one.hits, (r.hits, one.hits)
    dist.barrier()
    if rank == 0:
        print(f"nccl linkpred check ok on {world} GPUs: MRR {r.mrr:.6f}, Hits@10 {r.hits[10]:.6f}, {r.count} pairs")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
