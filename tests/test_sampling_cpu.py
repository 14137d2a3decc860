"""CPU side of the pair sampler: the oracle on a hand-computed graph of two components and an isolated node, the
uniformity of its destinations (chi-square, fixed seed), and PairSampler's epoch sources and rank shards - computed
with torch on the CPU - against the oracle and distributed.shard_indices' rule."""
import numpy as np
import pytest
import torch
from scipy.stats import chisquare

import sampling_oracle as so
from sympa_b200 import distributed as sd
from sympa_b200 import graphs
from sympa_b200.sampling import PairSampler, source_keys


def test_mix_is_splitmix64():
    # the first two outputs of the SplitMix64 generator seeded with 0
    assert so.mix(0) == 0xE220A8397B1DCDAF
    assert so.mix(0x9E3779B97F4A7C15) == 0x6E789E6AA1B965F4
    assert so.h(1, 2, 3, 4, 5) == so.mix(so.mix(so.mix(so.mix(so.mix(1) ^ 2) ^ 3) ^ 4) ^ 5)


def test_oracle_hand_computed_two_components():
    """path 0 - 1 - 2, edge 3 - 4, node 5 isolated:
    source 0 reaches [1, 2] at [1, 2] hops: draw k is node 1 + r with r = floor(2 h / 2^64), the top bit of h;
    source 3 reaches [4] only: every draw is (3, 4) at 1 hop;
    source 5 reaches nothing: (5, 5) at distance 0."""
    ptr, idx = graphs.adjacency_csr(torch.tensor([[0, 1], [1, 2], [3, 4]]), 6)
    seed, epoch, k = 7, 3, 6
    ids, d = so.sample_pairs(ptr.numpy(), idx.numpy(), [0, 3, 5, 2], k, seed, epoch)
    assert ids.shape == (4 * k, 2) and d.shape == (4 * k,)
    top = [so.h(seed, epoch, 0, 0, j) >> 63 for j in range(k)]
    assert 0 < sum(top) < k                                     # both destinations of source 0 occur
    assert ids[:k].tolist() == [[0, 1 + t] for t in top] and d[:k].tolist() == [1.0 + t for t in top]
    assert ids[k:2 * k].tolist() == [[3, 4]] * k and d[k:2 * k].tolist() == [1.0] * k
    assert ids[2 * k:3 * k].tolist() == [[5, 5]] * k and d[2 * k:3 * k].tolist() == [0.0] * k
    # source 2 reaches [0, 1] at [2, 1] hops
    top2 = [so.h(seed, epoch, 0, 2, j) >> 63 for j in range(k)]
    assert ids[3 * k:].tolist() == [[2, t] for t in top2] and d[3 * k:].tolist() == [2.0 - t for t in top2]
    # the draws of a source do not depend on the other sources or its position
    again, d2 = so.sample_pairs(ptr.numpy(), idx.numpy(), [2, 0], k, seed, epoch)
    assert again[:k].tolist() == ids[3 * k:].tolist() and again[k:].tolist() == ids[:k].tolist()


def test_destinations_are_uniform():
    """one source of a 10-node tree, 20 000 draws over its 9 reachable nodes: a chi-square test of uniformity (the
    draws are a fixed function of the seed, so the statistic is deterministic)"""
    ptr, idx = graphs.adjacency_csr(torch.tensor([[1, 0], [2, 0], [3, 1], [4, 1], [5, 2], [6, 5], [7, 5], [8, 7], [9, 3]]), 10)
    k = 20000
    ids, d = so.sample_pairs(ptr.numpy(), idx.numpy(), [5], k, seed=12345, epoch=0)
    counts = np.bincount(ids[:, 1], minlength=10)
    assert counts[5] == 0 and (counts[np.arange(10) != 5] > 0).all()
    stat, p = chisquare(counts[np.arange(10) != 5])
    assert p > 1e-3, (stat, p, counts)
    # the distances are the hop distances from node 5
    hops = {0: 2, 1: 3, 2: 1, 3: 4, 4: 4, 6: 1, 7: 1, 8: 2, 9: 5}
    assert all(d[i] == hops[int(ids[i, 1])] for i in range(0, k, 97))


def random_graph(n, seed):
    """a sparse random graph with isolated nodes (degree 0: never a source)"""
    rng = np.random.default_rng(seed)
    src = rng.integers(0, n - 8, 2 * n)
    dst = rng.integers(0, n - 8, 2 * n)
    return graphs.adjacency_csr(torch.from_numpy(np.stack((src, dst), 1)), n)


@pytest.mark.parametrize("seed", [0, 3, (1 << 64) - 5])
def test_source_keys_equal_the_oracle_hash(seed):
    nodes = torch.tensor([0, 1, 2, 77, (1 << 31) - 1, 1 << 40], dtype=torch.int64)
    for epoch in (0, 1, (1 << 64) - 1):
        got = source_keys(seed, epoch, nodes).tolist()
        want = [so.h(seed, epoch, 1, int(v), 0) for v in nodes]
        assert [(g + (1 << 63)) for g in got] == want     # signed order = unsigned order of the hash


@pytest.mark.parametrize("sources", [1, 13, 40])
def test_epoch_sources_equal_the_oracle(sources):
    ptr, idx = random_graph(64, 5)
    sampler = PairSampler((ptr, idx), sources, 3, seed=9)
    assert sampler.eligible.numel() < 64
    for epoch in (0, 1, 6):
        want = so.epoch_sources(ptr.numpy(), sources, 9, epoch)
        got = sampler.epoch_sources(epoch)
        assert got.dtype == torch.int64 and got.tolist() == want.tolist()
        assert len(set(want.tolist())) == sources and all(ptr[v + 1] > ptr[v] for v in want)
    if sources > 1:
        assert sampler.epoch_sources(0).tolist() != sampler.epoch_sources(1).tolist()


@pytest.mark.parametrize("sources,world", [(13, 1), (13, 2), (13, 4), (12, 3), (2, 3)])
def test_rank_shards_follow_shard_indices(sources, world):
    ptr, idx = random_graph(64, 6)
    sampler = PairSampler((ptr, idx), sources, 5, seed=2)
    full = sampler.epoch_sources(4)
    per = -(-sources // world)
    seen = []
    for rank in range(world):
        got = sampler.epoch_sources(4, rank, world)
        assert got.tolist() == full[sd.shard_indices(sources, rank, world, shuffle=False)].tolist()
        assert got.tolist() == so.epoch_sources(ptr.numpy(), sources, 2, 4, rank, world).tolist()
        assert got.numel() == per
        seen += got.tolist()
    assert sorted(set(seen)) == sorted(full.tolist())          # every source on some rank, padding by wrapping
    assert sampler.pairs_per_rank(world) == per * 5


def test_sampler_arguments():
    ptr, idx = random_graph(64, 7)
    eligible = int((ptr[1:] > ptr[:-1]).sum())
    with pytest.raises(ValueError, match="exceeds"):
        PairSampler((ptr, idx), eligible + 1, 4)
    PairSampler((ptr, idx), eligible, 4)
    with pytest.raises(ValueError):
        PairSampler((ptr, idx), 0, 4)
    with pytest.raises(ValueError):
        PairSampler((ptr, idx), 4, 0)
    with pytest.raises(ValueError):
        PairSampler((ptr.int(), idx), 4, 4)
    with pytest.raises(ValueError):
        PairSampler((ptr, idx), 4, 4, seed=-1)
    with pytest.raises(ValueError):
        PairSampler((ptr, idx), 4, 4).epoch_sources(1 << 64)
    with pytest.raises(RuntimeError, match="no CPU path"):
        PairSampler((ptr, idx), 4, 4).sample(0)
