"""CPU side of link-prediction evaluation: the numpy definition (rank_oracle) pinned on hand-checked rows, the edge
split of graphs.split_edges against a Python-integer hash oracle, and the argument checks of metrics.link_prediction,
which run before any launch."""
import numpy as np
import pytest
import torch

import rank_oracle
import sampling_oracle


def test_oracle_on_the_worked_example():
    # N = 6, u = 0, F(0) = {1}
    row = [0.0, 1.0, 2.0, 2.0, 2.0, 3.0]
    got = {v: rank_oracle.counts(row, 0, v, [1]) for v in (2, 5, 1)}
    assert got == {2: (0, 2), 5: (3, 3), 1: (0, 0)}
    rank, opt, pess = rank_oracle.ranks(*zip(*(got[v] for v in (2, 5, 1))))
    assert rank.tolist() == [2.0, 4.0, 1.0]
    assert opt.tolist() == [1.0, 4.0, 1.0]
    assert pess.tolist() == [3.0, 4.0, 1.0]


def test_oracle_on_signed_zeros_inf_and_repeats():
    # N = 7, u = 3, F(3) = {5}; -0.0 at column 0 equals +0.0 at column 4
    d = np.zeros((7, 7))
    d[3] = [-0.0, 0.5, np.inf, 0.0, 0.0, np.inf, 0.5]
    ptr = np.array([0, 0, 0, 0, 1, 1, 1, 1])
    idx = np.array([5])
    # a repeated pair (3, 2); the target 2 is listed twice for the same query
    pairs = [(3, 0), (3, 2), (3, 5), (3, 4), (3, 2)]
    lt, le = rank_oracle.pair_counts(d, pairs, ptr, idx)
    assert lt.tolist() == [0, 4, 4, 0, 4]
    assert le.tolist() == [1, 4, 5, 1, 4]
    rank, opt, pess = rank_oracle.ranks(lt, le)
    assert rank.tolist() == [1.5, 5.0, 5.5, 1.5, 5.0]
    assert opt.tolist() == [1.0, 5.0, 5.0, 1.0, 5.0] and pess.tolist() == [2.0, 5.0, 6.0, 2.0, 5.0]
    # a NaN anywhere in the row but the diagonal makes every pair of the row undefined
    d[3, 6] = np.nan
    lt, le = rank_oracle.pair_counts(d, pairs, ptr, idx)
    assert lt.tolist() == [-1] * 5 and le.tolist() == [-1] * 5
    assert np.isnan(rank_oracle.ranks(lt, le)[0]).all()
    d[3, 6] = 0.5
    d[3, 3] = np.nan
    lt, le = rank_oracle.pair_counts(d, pairs[:1], ptr, idx)        # the diagonal is not a competitor
    assert lt.tolist() == [0] and le.tolist() == [1]


def canonical(edges):
    return sorted({(min(a, b), max(a, b)) for a, b in edges if a != b})


def random_edges(rng, n, m):
    e = rng.integers(0, n, (m, 2))
    e[:5, 1] = e[:5, 0]                                   # self loops
    e = np.concatenate((e, e[10:20, ::-1], e[20:25]))     # flipped and repeated edges
    return torch.from_numpy(np.ascontiguousarray(e))


@pytest.mark.parametrize("seed,fraction", [(0, 0.1), (7, 0.5), (2 ** 64 - 1, 0.05), (3, 0.0), (4, 1.0)])
def test_split_edges_against_the_hash_oracle(seed, fraction):
    from sympa_b200 import graphs
    rng = np.random.default_rng(seed % 1000)
    n = 300
    edges = random_edges(rng, n, 900)
    train, test = graphs.split_edges(edges, n, fraction, seed=seed)
    canon = canonical(edges.tolist())
    held = round(fraction * len(canon))
    keyed = sorted(canon, key=lambda e: (sampling_oracle.h(seed, 0, 3, e[0], e[1]), e[0], e[1]))
    assert test.tolist() == [list(e) for e in sorted(keyed[:held])]
    assert train.tolist() == [list(e) for e in sorted(keyed[held:])]
    assert train.dtype == test.dtype == torch.int64 and train.shape[1] == test.shape[1] == 2
    again = graphs.split_edges(edges[torch.randperm(edges.shape[0], generator=torch.Generator().manual_seed(1))].flip(1),
                               n, fraction, seed=seed)
    assert torch.equal(again[0], train) and torch.equal(again[1], test)


def test_split_edges_is_the_same_on_cuda():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    from sympa_b200 import graphs
    edges = random_edges(np.random.default_rng(5), 5000, 20000)
    cpu = graphs.split_edges(edges, 5000, 0.1, seed=11)
    gpu = graphs.split_edges(edges.cuda(), 5000, 0.1, seed=11)
    assert gpu[0].is_cuda and torch.equal(gpu[0].cpu(), cpu[0]) and torch.equal(gpu[1].cpu(), cpu[1])


def test_split_edges_rejects_bad_input():
    from sympa_b200 import graphs
    e = torch.tensor([[0, 1], [1, 2]])
    for bad in (-0.1, 1.5):
        with pytest.raises(ValueError, match="test_fraction"):
            graphs.split_edges(e, 3, bad)
    with pytest.raises(ValueError, match="lie in"):
        graphs.split_edges(e, 2, 0.5)
    with pytest.raises(ValueError, match="int64"):
        graphs.split_edges(e.int(), 3, 0.5)
    train, test = graphs.split_edges(torch.zeros(0, 2, dtype=torch.int64), 3, 0.5)
    assert train.shape == test.shape == (0, 2)


def test_pair_keys_are_the_hash():
    from sympa_b200 import sampling
    u = torch.tensor([0, 5, 17, 2 ** 40])
    v = torch.tensor([1, 3, 17, 2 ** 33 + 1])
    got = sampling.source_keys(9, 4, u, tag=3, second=v)
    want = [sampling_oracle.h(9, 4, 3, a, b) - (1 << 63) for a, b in zip(u.tolist(), v.tolist())]
    assert got.tolist() == want
    # without a second argument: h(seed, epoch, tag, node, 0), as before
    assert torch.equal(sampling.source_keys(9, 4, u, tag=2), sampling.source_keys(9, 4, u, tag=2, second=torch.zeros_like(u)))


@pytest.fixture
def upper():
    from sympa_b200 import UpperHalfManifold, graphs
    man = UpperHalfManifold(dims=2)
    return man, man.random(10), graphs.adjacency_csr(torch.tensor([[0, 1], [1, 2]]), 10)


def test_link_prediction_checks_its_arguments(upper):
    from sympa_b200.metrics import link_prediction
    man, table, adj = upper
    ok = torch.tensor([[0, 1], [3, 4]])
    with pytest.raises(ValueError, match=r"pairs must lie in \[0, 10\)"):
        link_prediction(man, table, torch.tensor([[0, 10]]), adj)
    with pytest.raises(ValueError, match="pairs must lie"):
        link_prediction(man, table, torch.tensor([[-1, 2]]), adj)
    with pytest.raises(ValueError, match="u == v"):
        link_prediction(man, table, torch.tensor([[0, 1], [4, 4]]), adj)
    with pytest.raises(TypeError, match="int64"):
        link_prediction(man, table, ok.int(), adj)
    with pytest.raises(ValueError, match=r"\(E, 2\)"):
        link_prediction(man, table, torch.tensor([0, 1]), adj)
    for ks in ((0,), (1, -3)):
        with pytest.raises(ValueError, match="k of ks"):
            link_prediction(man, table, ok, adj, ks=ks)
    with pytest.raises(ValueError, match="N \\+ 1 row pointers"):
        link_prediction(man, table, ok, (adj[0][:-1], adj[1]))
    with pytest.raises(RuntimeError, match="no CPU path"):
        link_prediction(man, table, ok, adj)


def test_link_prediction_refuses_a_cpu_table_with_no_pairs(upper):
    from sympa_b200.metrics import link_prediction
    man, table, adj = upper
    with pytest.raises(RuntimeError, match="no CPU path"):
        link_prediction(man, table, torch.zeros(0, 2, dtype=torch.int64), adj)
