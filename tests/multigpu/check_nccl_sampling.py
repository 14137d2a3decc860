"""Multi-GPU (NCCL) check of sampled training pairs; run under torchrun on >= 2 GPUs, e.g.
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multigpu/check_nccl_sampling.py
(not collected by pytest).  Every rank samples its shard of the epoch's sources (sampling.PairSampler.sample with its
rank): the shards are disjoint and together equal one single-rank call.  One presharded FusedEpochRunner epoch on
those shards, gradients averaged over the ranks, leaves the same table on every rank."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def main():
    from types import SimpleNamespace

    from sympa_b200 import distributed as sd
    from sympa_b200 import graphs
    from sympa_b200.model import Model
    from sympa_b200.runner import FusedEpochRunner
    from sympa_b200.sampling import PairSampler

    rank, world, local = sd.init_process_group()
    dev = torch.device("cuda", local)
    ids, gd, n_nodes = graphs.product_cartesian_triplets(2, 2, 4, 2)
    adj = graphs.adjacency_csr(ids[gd == 1], n_nodes)
    adj = (adj[0].to(dev), adj[1].to(dev))
    sources, k = 2 * 57, 12                      # divisible by 2: the two shards are disjoint
    sampler = PairSampler(adj, sources, k, seed=4)
    one_ids, one_gd = sampler.sample(2)
    my_ids, my_gd = sampler.sample(2, rank, world)
    parts = [torch.empty_like(my_ids) for _ in range(world)]
    dist.all_gather(parts, my_ids)
    gparts = [torch.empty_like(my_gd) for _ in range(world)]
    dist.all_gather(gparts, my_gd)
    if sources % world == 0:
        mine = set(sampler.epoch_sources(2, rank, world).tolist())
        others = [set(p[::k, 0].tolist()) for p in parts]
        assert all(not (a & b) for i, a in enumerate(others) for b in others[i + 1:]), "rank shards overlap"
        assert others[rank] == mine
    # rank r holds sources r, r + world, ...: interleave the blocks back into the single-rank order
    per = -(-sources // world)
    blocks = torch.stack([p.reshape(per, k, 2) for p in parts], 1).reshape(per * world, k, 2)[:sources]
    gblocks = torch.stack([p.reshape(per, k) for p in gparts], 1).reshape(per * world, k)[:sources]
    assert torch.equal(blocks.reshape(-1, 2), one_ids) and torch.equal(gblocks.reshape(-1), one_gd)

    args = SimpleNamespace(manifold="upper", metric="riem", dims=3, num_points=n_nodes, scale_init=1.0, scale_coef=1.0,
                           train_scale=False)
    torch.manual_seed(0)
    model = Model(args).to(dev)
    runner = FusedEpochRunner(model, 1e-2 * world, my_ids, my_gd, 256, world_size=world, rank=rank, presharded=True)
    loss = runner.run_epoch(2)
    table = model.embeddings.embeds.detach()
    tables = [torch.empty_like(table) for _ in range(world)]
    dist.all_gather(tables, table)
    assert all(torch.equal(t, tables[0]) for t in tables), "tables differ between ranks"
    dist.barrier()
    if rank == 0:
        print(f"nccl sampling check ok on {world} GPUs: {one_ids.shape[0]} pairs, presharded epoch loss {loss:.6f}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
