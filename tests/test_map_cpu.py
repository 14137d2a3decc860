"""CPU side of the graph-reconstruction mAP: the CSR adjacency builder against networkx, and the numpy oracle
(closed form vs the argsort loop, and a hand-computed example with ties and a node without neighbours)."""
import networkx as nx
import numpy as np
import pytest
import torch

from map_oracle import ap_argsort_loop, ap_closed_form, ap_rows
from sympa_b200 import graphs


def _csr_of_networkx(g, n):
    ptr, idx = [0], []
    for u in range(n):
        nb = sorted(v for v in g.neighbors(u) if v != u)
        idx += nb
        ptr.append(len(idx))
    return ptr, idx


def _check(edges, n, g):
    ptr, idx = graphs.adjacency_csr(edges, n)
    want_ptr, want_idx = _csr_of_networkx(g, n)
    assert ptr.dtype == torch.int64 and idx.dtype == torch.int64
    assert ptr.tolist() == want_ptr
    assert idx.tolist() == want_idx


def test_adjacency_csr_grid():
    g = nx.convert_node_labels_to_integers(nx.grid_graph(dim=[4, 4]), ordering="sorted")
    ids, gd, n = graphs.grid_triplets(4, 2)
    assert n == g.number_of_nodes()
    # the grid generator orders nodes as itertools.product does: the same labels as the sorted networkx nodes
    _check(ids[gd == 1], n, g)


def test_adjacency_csr_tree_with_duplicates_and_self_loops():
    b, h = 3, 3
    g = nx.balanced_tree(b, h)
    n = g.number_of_nodes()
    k = torch.arange(1, n)
    edges = torch.stack((k, (k - 1) // b), 1)
    # duplicates, reversed duplicates and self loops must not change the result
    noisy = torch.cat((edges, edges[:7], edges[3:11].flip(1), torch.tensor([[0, 0], [5, 5], [n - 1, n - 1]])))
    noisy = noisy[torch.randperm(noisy.shape[0], generator=torch.Generator().manual_seed(0))]
    _check(noisy, n, g)
    _check(edges, n, g)


def test_adjacency_csr_product_graph():
    ids, gd, n = graphs.product_cartesian_triplets(2, 2, 3, 2)
    tree = nx.balanced_tree(2, 2)
    grid = nx.grid_graph(dim=[3, 3])
    g = nx.convert_node_labels_to_integers(nx.cartesian_product(tree, grid), ordering="sorted")
    assert n == g.number_of_nodes()
    _check(ids[gd == 1], n, g)


def test_adjacency_csr_isolated_nodes_and_bad_input():
    ptr, idx = graphs.adjacency_csr(torch.tensor([[1, 3]]), 5)
    assert ptr.tolist() == [0, 0, 1, 1, 2, 2] and idx.tolist() == [3, 1]
    ptr, idx = graphs.adjacency_csr(torch.zeros(0, 2, dtype=torch.int64), 3)
    assert ptr.tolist() == [0, 0, 0, 0] and idx.numel() == 0
    with pytest.raises(ValueError):
        graphs.adjacency_csr(torch.tensor([[0, 5]]), 5)
    with pytest.raises(ValueError):
        graphs.adjacency_csr(torch.tensor([0, 1]), 5)


def test_oracle_closed_form_equals_argsort_loop_without_ties():
    rng = np.random.default_rng(0)
    n = 60
    for trial in range(20):
        d = rng.random((n, n)) * 10 + 0.1
        for u in range(n):
            deg = int(rng.integers(0, 8))
            nbrs = rng.choice(np.delete(np.arange(n), u), size=deg, replace=False)
            a, b = ap_closed_form(d[u], u, nbrs), ap_argsort_loop(d[u], u, nbrs)
            if deg == 0:
                assert np.isnan(a) and np.isnan(b)
            else:
                assert abs(a - b) <= 1e-15 * max(abs(a), 1.0), (trial, u, a, b)


def test_oracle_hand_computed_ties_and_zero_degree():
    # node 0: d = (self, 1, 1, 2, 3), N(0) = {2, 3}: v = 2 -> 1 hit / 2 nodes at <= 1, v = 3 -> 2 / 3  => 7/12
    # node 1: d = (1, self, 1, 1, 5), N(1) = {0, 2}: both at 1, 2 hits / 3 nodes at <= 1 each      => 2/3
    # node 2: no neighbours                                                                      => NaN
    d = np.array([[0.0, 1, 1, 2, 3],
                  [1, 0.0, 1, 1, 5],
                  [1, 1, 0.0, 1, 1]])
    ptr = [0, 2, 4, 4, 4, 4]
    idx = [2, 3, 0, 2]
    ap = ap_rows(d, 0, ptr, idx)
    assert ap[0] == pytest.approx(7 / 12, rel=1e-15)
    assert ap[1] == pytest.approx(2 / 3, rel=1e-15)
    assert np.isnan(ap[2])
    assert np.nanmean(ap) == pytest.approx((7 / 12 + 2 / 3) / 2, rel=1e-15)
    # with ties the argsort loop depends on the tie order: the definition is its value when the tied
    # non-neighbours come first (here the stable order of row 0 puts node 1 before node 2)
    assert ap_argsort_loop(d[0], 0, [2, 3]) == pytest.approx(7 / 12, rel=1e-15)


def test_map_module_imports_without_a_gpu():
    from sympa_b200 import metrics
    assert callable(metrics.mean_average_precision)
    m = metrics.MeanAveragePrecisionMetric(graphs.adjacency_csr(torch.tensor([[0, 1]]), 2))
    assert m.adj[0].tolist() == [0, 1, 2]
    with pytest.raises(RuntimeError, match="no CPU path"):
        metrics.mean_average_precision(None, torch.zeros(2, 2, 1, 1, dtype=torch.float64), m.adj)

