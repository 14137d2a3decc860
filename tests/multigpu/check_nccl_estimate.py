"""Multi-GPU (NCCL) check of the sampled-row estimates; run under torchrun on >= 2 GPUs, e.g.
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multigpu/check_nccl_estimate.py
(not collected by pytest).  Every rank evaluates its distributed.row_shard part of the S sampled rows; the all-reduced
sums give estimates and standard errors that must equal the single-rank ones, and each rank's per-node values must be
its slice of the single-rank values."""
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
    from sympa_b200.metrics import estimate

    rank, world, local = sd.init_process_group()
    dev = torch.device("cuda", local)
    ids, gd, n_nodes = graphs.product_cartesian_triplets(2, 2, 4, 2)
    adj = graphs.adjacency_csr(ids[gd == 1], n_nodes)
    table = so.upper_spread(n_nodes, 3, generator=torch.Generator().manual_seed(0), scale=0.3).to(dev)
    man = UpperHalfManifold(dims=3, metric=MetricType.from_str("fone")).to(dev)
    kw = dict(scale=1.4, seed=5, epoch=1, block_bytes=12 * n_nodes * 5)
    rows = 101
    one = estimate(man, table, adj, rows, **kw)
    r = estimate(man, table, adj, rows, world_size=world, rank=rank, **kw)
    begin, end, _ = sd.row_shard(rows, rank, world)
    assert torch.equal(r.nodes, one.nodes[begin:end])
    assert torch.equal(torch.isnan(r.ap), torch.isnan(one.ap[begin:end]))
    assert torch.equal(r.ap.nan_to_num(), one.ap[begin:end].nan_to_num())
    for a, b in zip(r.distortion, one.distortion):
        assert torch.equal(a, b[begin:end])
    for name in ("mean_ap", "mean_ap_se", "average_distortion", "average_distortion_se"):
        x, y = getattr(r, name), getattr(one, name)
        assert y > 0 and abs(x - y) <= 1e-13 * y, (name, x, y)
    assert r.sampled_worst_case_distortion == one.sampled_worst_case_distortion
    dist.barrier()
    if rank == 0:
        print(f"nccl estimate check ok on {world} GPUs: mAP {r.mean_ap:.6f} +- {r.mean_ap_se:.6f}, "
              f"average distortion {r.average_distortion:.6f} +- {r.average_distortion_se:.6f}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
