"""CPU side of the exact k-nearest-neighbour queries: the numpy definition (knn_oracle) pinned on a hand-computed
example, and the argument checks of metrics.nearest, which run before any launch."""
import numpy as np
import pytest
import torch

import knn_oracle

# ties across columns (1.0 at 1 and 4), -0.0 next to +0.0 (columns 5 and 3), a NaN (column 2)
ROW = [3.0, 1.0, np.nan, 0.0, 1.0, -0.0, 2.0]


def test_oracle_on_a_hand_computed_row():
    block = np.array([ROW, ROW])
    # row 0 leaves nothing out: 6 selectable entries; row 1 leaves out column 1: 5 selectable entries
    ids, vals = knn_oracle.topk(block, 6, exclude=[-1, 1])
    assert ids.tolist() == [[3, 5, 1, 4, 6, 0], [3, 5, 4, 6, 0, -1]]
    assert vals[0].tolist() == [0.0, 0.0, 1.0, 1.0, 2.0, 3.0]
    assert np.signbit(vals[0]).tolist() == [False, True, False, False, False, False]    # -0.0 kept as stored
    assert vals[1, :5].tolist() == [0.0, 0.0, 1.0, 2.0, 3.0] and np.isnan(vals[1, 5])
    # k equal to the number of selectable entries, then one more
    ids, vals = knn_oracle.topk(block[:1], 6)
    assert ids.tolist() == [[3, 5, 1, 4, 6, 0]] and not np.isnan(vals).any()
    ids, vals = knn_oracle.topk(block[:1], 7)
    assert ids.tolist() == [[3, 5, 1, 4, 6, 0, -1]] and np.isnan(vals[0, 6])
    ids, vals = knn_oracle.topk(block[1:], 5, exclude=[1])
    assert ids.tolist() == [[3, 5, 4, 6, 0]]
    ids, vals = knn_oracle.topk(block[1:], 2, exclude=[3])
    assert ids.tolist() == [[5, 1]] and np.signbit(vals[0, 0])


def test_oracle_is_the_stable_torch_sort():
    rng = np.random.default_rng(0)
    block = rng.integers(0, 4, (9, 40)).astype(np.float64) * 0.5
    block[2, 5] = np.nan
    block[3] = np.nan
    exclude = rng.integers(-1, 40, 9)
    ids, vals = knn_oracle.topk(block, 12, exclude=exclude)
    for r in range(9):
        keep = torch.arange(40)
        keep = keep[keep != int(exclude[r])]
        s = torch.sort(torch.from_numpy(block[r])[keep], stable=True)
        want_ids = keep[s.indices][:12].numpy().copy()
        want_vals = s.values[:12].numpy()
        want_ids[np.isnan(want_vals)] = -1
        assert ids[r].tolist() == want_ids.tolist()
        assert np.array_equal(vals[r], want_vals, equal_nan=True)


@pytest.fixture
def upper():
    from sympa_b200 import UpperHalfManifold
    man = UpperHalfManifold(dims=2)
    return man, man.random(10)


def test_nearest_checks_k(upper):
    from sympa_b200.metrics import nearest
    man, table = upper
    q = torch.tensor([0, 3], dtype=torch.int64)
    for k in (0, -1, 10, 1025):
        with pytest.raises(ValueError, match="k must lie in"):
            nearest(man, table, q, k)
    with pytest.raises(RuntimeError, match="no CPU path"):        # k = N is allowed when the node itself counts
        nearest(man, table, q, 10, exclude_self=False)
    with pytest.raises(ValueError, match="no neighbour"):
        nearest(man, table[:1], torch.tensor([0]), 1)


def test_nearest_checks_queries(upper):
    from sympa_b200.metrics import nearest
    man, table = upper
    with pytest.raises(ValueError, match=r"queries must lie in \[0, 10\)"):
        nearest(man, table, torch.tensor([0, 10]), 3)
    with pytest.raises(ValueError, match="queries must lie"):
        nearest(man, table, torch.tensor([-1]), 3)
    with pytest.raises(TypeError, match="int64"):
        nearest(man, table, torch.tensor([0, 1], dtype=torch.int32), 3)
    with pytest.raises(TypeError, match="int64"):
        nearest(man, table, [0, 1], 3)
    with pytest.raises(ValueError, match="1-D"):
        nearest(man, table, torch.zeros(2, 2, dtype=torch.int64), 3)


def test_nearest_refuses_a_cpu_table(upper):
    from sympa_b200.metrics import nearest
    man, table = upper
    with pytest.raises(RuntimeError, match="no CPU path"):
        nearest(man, table, torch.tensor([1, 1, 4]), 3)
    with pytest.raises(RuntimeError, match="no CPU path"):
        nearest(man, table, torch.empty(0, dtype=torch.int64), 3)
