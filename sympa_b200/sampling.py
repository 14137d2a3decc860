"""Training pairs sampled from an edge list, for graphs whose all-pairs triplets do not fit in memory.

Every epoch draws `sources_per_epoch` sources and `pairs_per_source` destinations per source, each with its hop
distance, by breadth-first search on the GPU (ops.sample_pairs).  The result is the (src_dst_ids, graph_distances)
pair of tensors that runner.train_epoch and runner.FusedEpochRunner already take.  The rule, which a CPU oracle
reproduces bit for bit:

  mix        the SplitMix64 finalizer, h(seed, epoch, tag, a, b) = mix(mix(mix(mix(mix(seed) ^ epoch) ^ tag) ^ a) ^ b)
  sources    the nodes of degree >= 1 sorted by (h(seed, epoch, 1, node, 0), node); the first sources_per_epoch
  shards     rank r of P takes positions r, r + P, ... of that list, padded by wrapping to P ceil(S / P)
             (distributed.shard_indices without shuffling), so every rank gets the same number of pairs
  pairs      draw k of source u: uniform over the nodes u reaches, from h(seed, epoch, 0, u, k)
             (sympa_sample_pairs in include/sympa_b200.h)

    sampler = PairSampler(adj, sources_per_epoch=4096, pairs_per_source=256, seed=0)
    ids, gd = sampler.sample(0)
    runner = FusedEpochRunner(model, lr, ids, gd, batch_size)
    for epoch in range(epochs):
        sampler.sample(epoch, out=(runner.ids, runner.gdist))     # fresh pairs in the runner's own tensors
        runner.run_epoch(epoch)
"""
import torch

from . import distributed as sd
from . import ops

_M64 = (1 << 64) - 1


def _mix(x):
    """the SplitMix64 finalizer on a Python integer"""
    x = (x + 0x9E3779B97F4A7C15) & _M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & _M64
    return x ^ (x >> 31)


def _i64(v):
    """the int64 with the bits of the uint64 v"""
    return v - (1 << 64) if v >= 1 << 63 else v


def _shr(x, s):
    """logical right shift of an int64 tensor read as uint64"""
    return (x >> s) & ((1 << (64 - s)) - 1)


def _mix_tensor(x):
    """the SplitMix64 finalizer on an int64 tensor read as uint64 (int64 addition and multiplication wrap mod 2^64)"""
    x = x + _i64(0x9E3779B97F4A7C15)
    x = (x ^ _shr(x, 30)) * _i64(0xBF58476D1CE4E5B9)
    x = (x ^ _shr(x, 27)) * _i64(0x94D049BB133111EB)
    return x ^ _shr(x, 31)


def source_keys(seed, epoch, nodes, tag=1, second=None):
    """h(seed, epoch, tag, node, 0) of every node of the int64 tensor `nodes`, or h(seed, epoch, tag, node, b) with b
    the matching entry of the int64 tensor `second`, as int64 tensors whose signed order is the unsigned order of the
    hash.  Tag 1 orders the training sources, tag 2 the nodes metrics.estimate samples, tag 3 (with the second
    endpoint) the edges graphs.split_edges holds out."""
    head = _i64(_mix(_mix(_mix(seed) ^ epoch) ^ tag))
    h = _mix_tensor(nodes ^ head)
    h = _mix_tensor(h if second is None else h ^ second)
    return h ^ _i64(1 << 63)


class PairSampler:
    """Training pairs of the undirected graph adj = (ptr, idx) (graphs.adjacency_csr), drawn per epoch by the rule of
    the module docstring.  adj on a CUDA device for sample(); epoch_sources() runs on adj's device, CPU included."""

    def __init__(self, adj, sources_per_epoch, pairs_per_source, seed=0):
        ptr, idx = adj
        if not (isinstance(ptr, torch.Tensor) and isinstance(idx, torch.Tensor)) or ptr.dtype != torch.int64 \
                or idx.dtype != torch.int64 or ptr.dim() != 1 or ptr.numel() < 1 or idx.dim() != 1:
            raise ValueError("adj must be (ptr, idx): 1-D int64 tensors, ptr with N + 1 entries")
        if idx.device != ptr.device:
            raise ValueError("adjacency ptr and idx must be on the same device")
        self.adj = (ptr.contiguous(), idx.contiguous())
        self.num_nodes = ptr.numel() - 1
        self.sources_per_epoch, self.pairs_per_source, self.seed = int(sources_per_epoch), int(pairs_per_source), int(seed)
        if not 0 <= self.seed < 1 << 64:
            raise ValueError("seed must lie in [0, 2^64)")
        if self.sources_per_epoch < 1 or self.pairs_per_source < 1:
            raise ValueError("sources_per_epoch and pairs_per_source must be >= 1")
        # after adjacency_csr removes self loops, exactly the nodes that reach another node
        self.eligible = torch.nonzero(ptr[1:] > ptr[:-1]).reshape(-1)
        if self.sources_per_epoch > self.eligible.numel():
            raise ValueError(f"sources_per_epoch = {self.sources_per_epoch} exceeds the {self.eligible.numel()} nodes "
                             "with at least one neighbour")

    def pairs_per_rank(self, world_size=1):
        """rows of sample(..., world_size=world_size): ceil(S / world_size) sources of pairs_per_source pairs each"""
        return -(-self.sources_per_epoch // world_size) * self.pairs_per_source

    def epoch_sources(self, epoch, rank=0, world_size=1):
        """the sources of `epoch` that rank `rank` of `world_size` samples, as an int64 tensor on adj's device"""
        epoch = int(epoch)
        if not 0 <= epoch < 1 << 64:
            raise ValueError("epoch must lie in [0, 2^64)")
        order = torch.sort(source_keys(self.seed, epoch, self.eligible), stable=True).indices   # ties: by node
        chosen = self.eligible[order[: self.sources_per_epoch]]
        return chosen[sd.shard_indices(self.sources_per_epoch, rank, world_size, shuffle=False, device=chosen.device)]

    def sample(self, epoch, rank=0, world_size=1, out=None):
        """(src_dst_ids (pairs_per_rank, 2) int64, graph_distances (pairs_per_rank,) float64) of this rank's sources
        of `epoch`; out = (ids, gd) to write into.  Pass presharded=True to the trainer when world_size > 1."""
        return ops.sample_pairs(self.adj, self.epoch_sources(epoch, rank, world_size), self.pairs_per_source, self.seed,
                                epoch, out=out)
