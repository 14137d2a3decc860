"""CPU side of the graph-reconstruction distortion: scipy's hop distances against the closed-form triplet
generators, the oracle on a hand-computed example (a second component, a scale != 1, a NaN distance), and the
metrics refusing a CPU table."""
import numpy as np
import pytest
import torch

from distortion_oracle import distortion, distortion_rows, hop_matrix
from sympa_b200 import graphs


@pytest.mark.parametrize("name,args", [("grid", (4, 2)), ("grid", (3, 3)), ("tree", (2, 3)), ("tree", (3, 2)),
                                       ("product", (2, 1, 3, 2)), ("product", (2, 2, 2, 2))])
def test_scipy_hop_distances_equal_the_generators(name, args):
    gen = {"grid": graphs.grid_triplets, "tree": graphs.balanced_tree_triplets,
           "product": graphs.product_cartesian_triplets}[name]
    ids, gd, n = gen(*args)
    ptr, idx = graphs.adjacency_csr(ids[gd == 1], n)
    h = hop_matrix(ptr.numpy(), idx.numpy())
    assert h.dtype == np.int32 and h.shape == (n, n)
    assert np.all(np.diag(h) == 0)
    i, j = ids[:, 0].numpy(), ids[:, 1].numpy()
    np.testing.assert_array_equal(h[i, j], gd.numpy().astype(np.int32))
    np.testing.assert_array_equal(h, h.T)
    # a row subset is the same rows
    np.testing.assert_array_equal(hop_matrix(ptr.numpy(), idx.numpy(), rows=np.arange(2, 5)), h[2:5])


def hand_example():
    """path 0 - 1 - 2 and the edge 3 - 4 (two components), scale 2:
    (0, 1): g 1, d 0.5,  s d 1   -> delta 0,   ratio 1
    (0, 2): g 2, d 1.5,  s d 3   -> delta 1/2, ratio 3/2
    (1, 2): g 1, d 0.25, s d 1/2 -> delta 1/2, ratio 1/2
    (3, 4): g 1, d 1,    s d 2   -> delta 1,   ratio 2
    average (0 + 1/2 + 1/2 + 1) / 4 = 1/2, worst case 2 / (1/2) = 4.  Pairs across the components (one of them
    NaN) and the lower triangle (u > w) are not read."""
    ptr, idx = graphs.adjacency_csr(torch.tensor([[0, 1], [1, 2], [3, 4]]), 5)
    d = np.full((5, 5), 7.0)
    np.fill_diagonal(d, 0.0)
    d[0, 1], d[0, 2], d[1, 2], d[3, 4] = 0.5, 1.5, 0.25, 1.0
    d[0, 4] = np.nan
    return ptr.numpy(), idx.numpy(), d, 2.0


def test_oracle_hand_computed_example():
    ptr, idx, d, s = hand_example()
    h = hop_matrix(ptr, idx)
    assert h[0].tolist() == [0, 1, 2, -1, -1] and h[3].tolist() == [-1, -1, -1, 0, 1]
    total, count, hi, lo = distortion_rows(d, h, 0, s)
    assert total.tolist() == [0.5, 0.5, 0.0, 1.0, 0.0]
    assert count.tolist() == [2, 1, 0, 1, 0]
    assert hi.tolist() == [1.5, 0.5, -np.inf, 2.0, -np.inf]
    assert lo.tolist() == [1.0, 0.5, np.inf, 2.0, np.inf]
    assert total.sum() / count.sum() == 0.5
    assert hi.max() / lo.min() == 4.0
    # the route over triplets gives the same two figures
    pairs = np.array([[0, 1], [0, 2], [1, 2], [3, 4]])
    avg, worst = distortion(s * d[pairs[:, 0], pairs[:, 1]], h[pairs[:, 0], pairs[:, 1]])
    assert (avg, worst) == (0.5, 4.0)
    # a row block starting at an offset holds the same rows
    part = distortion_rows(d[3:5], h[3:5], 3, s)
    assert part[0].tolist() == [1.0, 0.0] and part[1].tolist() == [1, 0]


def test_oracle_nan_distance_poisons_its_row_only():
    ptr, idx, d, s = hand_example()
    h = hop_matrix(ptr, idx)
    d[1, 2] = np.nan
    total, count, hi, lo = distortion_rows(d, h, 0, s)
    assert np.isnan(total[1]) and np.isnan(hi[1]) and np.isnan(lo[1]) and count[1] == 1
    assert total[0] == 0.5 and total[3] == 1.0


def test_distortion_metrics_refuse_a_cpu_table():
    from sympa_b200 import metrics
    adj = graphs.adjacency_csr(torch.tensor([[0, 1]]), 2)
    table = torch.zeros(2, 2, 1, 1, dtype=torch.float64)
    with pytest.raises(RuntimeError, match="no CPU path"):
        metrics.average_distortion(None, table, adj)
    with pytest.raises(RuntimeError, match="no CPU path"):
        metrics.evaluate(None, table, adj, scale=2.0)
