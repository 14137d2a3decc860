"""Python-integer / numpy oracle of the pair sampler (sympa_sample_pairs, sympa_b200.sampling), restating the rule of
include/sympa_b200.h independently of the package: SplitMix64 hashes in Python integers, hop distances from scipy's
csgraph."""
import numpy as np

from distortion_oracle import hop_matrix

M64 = (1 << 64) - 1


def mix(x):
    x = (x + 0x9E3779B97F4A7C15) & M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & M64
    return x ^ (x >> 31)


def h(seed, epoch, tag, a, b):
    return mix(mix(mix(mix(mix(seed) ^ epoch) ^ tag) ^ a) ^ b)


def draw_index(seed, epoch, u, k, c):
    """r = floor(h(seed, epoch, 0, u, k) * c / 2^64): the rank of draw k of source u among its c reachable nodes"""
    return (h(seed, epoch, 0, u, k) * c) >> 64


def pairs_from_rows(hop_rows, sources, k, seed, epoch):
    """(ids (S k, 2) int64, distances (S k,) float64) of the sources, hop_rows[i] the hop row of sources[i] (-1 where
    unreachable); a source that reaches no other node gets k pairs (u, u) at distance 0"""
    ids = np.zeros((len(sources) * k, 2), dtype=np.int64)
    dist = np.zeros(len(sources) * k)
    for i, u in enumerate(sources):
        u = int(u)
        reach = np.flatnonzero(hop_rows[i] >= 1)           # R(u) \ {u}, ascending node id
        for j in range(k):
            row = i * k + j
            if reach.size == 0:
                ids[row] = (u, u)
                continue
            dst = int(reach[draw_index(seed, epoch, u, j, reach.size)])
            ids[row] = (u, dst)
            dist[row] = float(hop_rows[i][dst])
    return ids, dist


def sample_pairs(ptr, idx, sources, k, seed, epoch):
    """what ops.sample_pairs returns for sources in [0, N)"""
    sources = np.asarray(sources, dtype=np.int64)
    if sources.size == 0:
        return np.zeros((0, 2), dtype=np.int64), np.zeros(0)
    uniq, inv = np.unique(sources, return_inverse=True)
    rows = hop_matrix(ptr, idx, rows=uniq)[inv]
    return pairs_from_rows(rows, sources, k, seed, epoch)


def epoch_sources(ptr, sources_per_epoch, seed, epoch, rank=0, world_size=1):
    """the nodes of degree >= 1 sorted by (h(seed, epoch, 1, node, 0), node), the first S of them; rank r of P takes
    positions r, r + P, ... of that list padded by wrapping to P ceil(S / P)"""
    ptr = np.asarray(ptr)
    eligible = [v for v in range(ptr.size - 1) if ptr[v + 1] > ptr[v]]
    if sources_per_epoch > len(eligible):
        raise ValueError("more sources than nodes with a neighbour")
    chosen = sorted(eligible, key=lambda v: (h(seed, epoch, 1, v, 0), v))[:sources_per_epoch]
    per = -(-sources_per_epoch // world_size)
    padded = [chosen[i % sources_per_epoch] for i in range(per * world_size)]
    return np.array(padded[rank::world_size], dtype=np.int64)
