"""Multi-GPU (NCCL) check of the row-sharded distortion evaluation; run under torchrun on >= 2 GPUs, e.g.
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multigpu/check_nccl_distortion.py
(not collected by pytest).  Every rank evaluates its distributed.row_shard rows of the distance matrix, and one
all-reduce of (sum, count) plus one MAX and one MIN give the global distortion, which must equal the single-rank
value; metrics.evaluate shares the same pass with mAP."""
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
    from sympa_b200.metrics import average_distortion, evaluate

    rank, world, local = sd.init_process_group()
    dev = torch.device("cuda", local)
    ids, gd, n_nodes = graphs.product_cartesian_triplets(2, 2, 4, 2)
    adj = graphs.adjacency_csr(ids[gd == 1], n_nodes)
    table = so.upper_spread(n_nodes, 3, generator=torch.Generator().manual_seed(0), scale=0.3).to(dev)
    man = UpperHalfManifold(dims=3, metric=MetricType.from_str("fone")).to(dev)
    kw = dict(scale=1.4, block_bytes=12 * n_nodes * 5)
    s1, c1, hi1, lo1, rows1 = average_distortion(man, table, adj, **kw)
    s, c, hi, lo, rows = average_distortion(man, table, adj, world_size=world, rank=rank, **kw)
    begin, end, _ = sd.row_shard(n_nodes, rank, world)
    assert rows.sum.shape == (end - begin,)
    for a, b in zip(rows, rows1):
        assert torch.equal(a, b[begin:end])
    assert c == c1 == ids.shape[0], (c, c1)
    assert abs(s / c - s1 / c1) <= 1e-15 * (s1 / c1), (s / c, s1 / c1)
    assert (hi, lo) == (hi1, lo1)
    r1 = evaluate(man, table, adj, **kw)
    r = evaluate(man, table, adj, world_size=world, rank=rank, **kw)
    assert abs(r.average_distortion - r1.average_distortion) <= 1e-15 * r1.average_distortion
    assert r.worst_case_distortion == r1.worst_case_distortion
    assert abs(r.mean_ap - r1.mean_ap) <= 1e-15
    assert torch.equal(r.ap, r1.ap[begin:end])
    dist.barrier()
    if rank == 0:
        print(f"nccl distortion check ok on {world} GPUs: average distortion {s / c:.15f}, "
              f"worst case {r.worst_case_distortion:.15f}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
