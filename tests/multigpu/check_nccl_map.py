"""Multi-GPU (NCCL) check of the row-sharded mAP evaluation; run under torchrun on >= 2 GPUs, e.g.
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multigpu/check_nccl_map.py
(not collected by pytest).  Every rank evaluates its distributed.row_shard rows of the distance matrix and one
all-reduce of (sum_ap, count) gives the global mAP, which must equal the single-rank value."""
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
    from sympa_b200.metrics import mean_average_precision

    rank, world, local = sd.init_process_group()
    dev = torch.device("cuda", local)
    ids, gd, n_nodes = graphs.product_cartesian_triplets(2, 2, 4, 2)
    adj = graphs.adjacency_csr(ids[gd == 1], n_nodes)
    table = so.upper_spread(n_nodes, 3, generator=torch.Generator().manual_seed(0), scale=0.3).to(dev)
    man = UpperHalfManifold(dims=3, metric=MetricType.from_str("fone")).to(dev)
    s1, c1, ap1 = mean_average_precision(man, table, adj, block_bytes=8 * n_nodes * 5)
    s, c, ap = mean_average_precision(man, table, adj, block_bytes=8 * n_nodes * 5, world_size=world, rank=rank)
    begin, end, _ = sd.row_shard(n_nodes, rank, world)
    assert ap.shape == (end - begin,)
    assert torch.equal(ap, ap1[begin:end])
    assert c == c1 == n_nodes, (c, c1)
    assert abs(s / c - s1 / c1) <= 1e-15, (s / c, s1 / c1)
    dist.barrier()
    if rank == 0:
        print(f"nccl map check ok on {world} GPUs: mAP {s / c:.15f}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
