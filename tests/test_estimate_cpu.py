"""CPU side of the sampled-row estimates (sympa_b200.metrics.estimate): the sample against a Python-integer evaluation
of the hash rule, source_keys' default tag unchanged, the relabelled CSR adjacency against the original graph under
the permutation (scipy), and the estimator and standard-error formulas against a two-pass numpy oracle."""
import math

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import sampling_oracle as so
from sympa_b200 import graphs
from sympa_b200.metrics import _estimates, sample_order
from sympa_b200.sampling import source_keys


@pytest.mark.parametrize("n,s,seed,epoch", [(1, 1, 0, 0), (37, 5, 3, 0), (200, 200, 11, 4), (1000, 64, (1 << 64) - 1, 9)])
def test_sample_order_is_the_hash_rule(n, s, seed, epoch):
    chosen = sorted(range(n), key=lambda v: (so.h(seed, epoch, 2, v, 0), v))[:s]
    rest = sorted(set(range(n)) - set(chosen))
    got = sample_order(n, s, seed=seed, epoch=epoch)
    assert got.dtype == torch.int64 and got.tolist() == chosen + rest


def test_the_sample_does_not_depend_on_its_size_or_the_training_sources():
    n = 500
    big = sample_order(n, 100, seed=5, epoch=2)
    assert sample_order(n, 30, seed=5, epoch=2)[:30].tolist() == big[:30].tolist()     # nested samples
    train = sorted(range(n), key=lambda v: (so.h(5, 2, 1, v, 0), v))[:30]
    assert big[:30].tolist() != train                                                   # tag 2, not tag 1


def test_source_keys_default_tag_is_unchanged():
    nodes = torch.arange(300, dtype=torch.int64)
    for seed, epoch in ((0, 0), (7, 3), ((1 << 64) - 1, (1 << 64) - 1)):
        keys = source_keys(seed, epoch, nodes)
        assert torch.equal(keys, source_keys(seed, epoch, nodes, tag=1))
        # h(seed, epoch, 1, node, 0) with its top bit flipped, read as int64: signed order = unsigned order of h
        want = [((so.h(seed, epoch, 1, v, 0) ^ (1 << 63)) + (1 << 63)) % (1 << 64) - (1 << 63) for v in range(300)]
        assert keys.tolist() == want
        want2 = [((so.h(seed, epoch, 2, v, 0) ^ (1 << 63)) + (1 << 63)) % (1 << 64) - (1 << 63) for v in range(300)]
        assert source_keys(seed, epoch, nodes, tag=2).tolist() == want2


def random_graph(n, seed):
    """a sparse random graph with isolated nodes and a hub"""
    rng = np.random.default_rng(seed)
    src = np.repeat(np.arange(n), rng.integers(0, 4, n))
    e = np.stack((src, rng.integers(0, n, src.size)), 1)
    e = np.concatenate((e, np.stack((np.zeros(n // 3, dtype=np.int64), np.arange(n // 3) * 3), 1)))
    return graphs.adjacency_csr(torch.from_numpy(e.astype(np.int64)), n)


@pytest.mark.parametrize("n", [1, 2, 97, 1500])
def test_relabelled_csr_is_the_graph_under_the_permutation(n):
    ptr, idx = random_graph(n, n)
    perm = torch.from_numpy(np.random.default_rng(n + 1).permutation(n).astype(np.int64))
    new_ptr, new_idx = graphs.relabel_csr((ptr, idx), perm)
    assert new_ptr.dtype == torch.int64 and new_idx.dtype == torch.int64 and new_ptr.shape == (n + 1,)
    a = sp.csr_matrix((np.ones(idx.numel()), idx.numpy(), ptr.numpy()), shape=(n, n))
    b = sp.csr_matrix((np.ones(new_idx.numel()), new_idx.numpy(), new_ptr.numpy()), shape=(n, n))
    p = perm.numpy()
    assert (b != a[p][:, p]).nnz == 0 and b.nnz == a.nnz
    # row i is row perm[i] with its entries renamed, in their old order
    inv = np.argsort(p)
    for i in range(0, n, max(1, n // 50)):
        old = idx[ptr[p[i]]:ptr[p[i] + 1]].numpy()
        assert new_idx[new_ptr[i]:new_ptr[i + 1]].tolist() == inv[old].tolist()


def test_relabel_with_the_sample_order_puts_the_sample_first():
    n = 300
    ptr, idx = random_graph(n, 4)
    perm = sample_order(n, 40, seed=1, epoch=0)
    new_ptr, _ = graphs.relabel_csr((ptr, idx), perm)
    deg, new_deg = (ptr[1:] - ptr[:-1]), (new_ptr[1:] - new_ptr[:-1])
    assert torch.equal(new_deg, deg[perm])


def oracle(ap, a, c, n_nodes, with_neighbours):
    """two-pass numpy evaluation of the module docstring's formulas over all S sampled rows"""
    s = a.size
    v = ap[~np.isnan(ap)]
    m = v.size
    mean_ap = v.mean()
    ap_se = v.std(ddof=1) / math.sqrt(m) * math.sqrt(1 - m / with_neighbours)
    r = a.sum() / c.sum()
    c_bar = c.mean()
    r_se = math.sqrt((1 - s / n_nodes) * ((a - r * c) ** 2).sum() / ((s - 1) * s * c_bar ** 2))
    return mean_ap, ap_se, r, r_se


def run(ap, a, c, n_nodes, with_neighbours, shards=1):
    """_estimates over `shards` row shards, their squared deviations summed as an all-reduce would"""
    ap_t, a_t, c_t = torch.tensor(ap), torch.tensor(a), torch.tensor(c, dtype=torch.int64)
    valid = ~np.isnan(ap)
    sums = (float(ap[valid].sum()), int(valid.sum()), float(a.sum()), float(c.sum()))
    if shards == 1:
        return _estimates(sums, ap_t, a_t, c_t, a.size, n_nodes, with_neighbours)
    parts = np.array_split(np.arange(a.size), shards)
    acc = []

    def reduce(t):                      # collects every shard's deviations; the last call sees their sum
        acc.append(t.clone())
        t.copy_(torch.stack(acc).sum(0))

    for k in parts:
        out = _estimates(sums, ap_t[k], a_t[k], c_t[k], a.size, n_nodes, with_neighbours, reduce)
    return out


def test_estimates_match_the_two_pass_oracle():
    # S = 6 sampled rows of N = 20 nodes, M = 15 of which have neighbours; row 1 is a node without neighbours
    ap = np.array([0.5, np.nan, 1.0, 0.25, 0.8, 2 / 3])
    a = np.array([1.25, 0.0, 3.0, 0.5, 2.2, 1.1])
    c = np.array([3, 0, 5, 2, 4, 4])
    want = oracle(ap, a, c, 20, 15)
    # by hand: mAP = (0.5 + 1 + 0.25 + 0.8 + 2/3) / 5, R = 8.05 / 18
    assert want[0] == pytest.approx((0.5 + 1 + 0.25 + 0.8 + 2 / 3) / 5, rel=1e-15) and want[2] == pytest.approx(8.05 / 18)
    for shards in (1, 2, 3):
        got = run(ap, a, c, 20, 15, shards)
        np.testing.assert_allclose(got, want, rtol=1e-14, atol=0)


def test_standard_errors_vanish_when_every_row_is_sampled():
    ap = np.array([0.5, np.nan, 1.0, 0.25])
    a = np.array([1.25, 0.0, 3.0, 0.5])
    c = np.array([3, 0, 5, 2])
    mean_ap, ap_se, r, r_se = run(ap, a, c, 4, 3)
    assert ap_se == 0.0 and r_se == 0.0
    assert mean_ap == pytest.approx(1.75 / 3, rel=1e-15) and r == pytest.approx(4.75 / 10, rel=1e-15)
    # one unit short of the population: a standard error needs two units
    assert all(math.isnan(x) for x in (run(ap[:1], a[:1], c[:1], 4, 3)[1], run(ap[:1], a[:1], c[:1], 4, 3)[3]))
