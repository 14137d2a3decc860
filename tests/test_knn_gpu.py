"""Exact k-nearest-neighbour queries on the device (sympa_dist_rows, sympa_row_topk, sympa_b200.metrics.nearest):
the selection kernel bit for bit against the numpy definition (knn_oracle) on blocks with heavy ties, -0.0, NaN and
rows long enough to be split over many CTAs; query rows bit-identical to the rows of dist_matrix; nearest equal to
the stable sort of the distance matrix rows, invariant to the block size and the rank shards; bounded memory and
the model's own scale."""
import types

import numpy as np
import pytest
import torch

import knn_oracle
import siegel_oracle as so

pytestmark = pytest.mark.gpu

METRICS = ["riem", "fone", "finf", "fmin", "wsum"]


@pytest.fixture(scope="module")
def sb():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    import sympa_b200
    import sympa_b200.metrics  # noqa: F401
    from sympa_b200 import _lib
    _lib.load()
    return sympa_b200


def bits(t):
    """the float64 tensor's bit patterns (so that NaN == NaN and -0.0 != +0.0)"""
    return t.detach().cpu().contiguous().view(torch.int64)


def assert_topk(got, want):
    ids, vals = got
    assert ids.cpu().tolist() == want[0].tolist()
    assert torch.equal(bits(vals), torch.from_numpy(np.ascontiguousarray(want[1])).view(torch.int64))


def status_bits(sb):
    from sympa_b200 import ops
    w = ops.status_word(torch.device("cuda", torch.cuda.current_device()))
    v = int(w.item())
    w.zero_()
    return v


def synthetic_blocks(rng):
    """(name, block) of heavy ties, all-equal rows, signed zeros, NaN entries and whole NaN rows"""
    levels = rng.integers(0, 5, (37, 3000)).astype(np.float64) * 0.25 - 0.5       # values from five levels
    levels[levels == 0.0] = np.where(rng.random((levels == 0.0).sum()) < 0.5, -0.0, 0.0)
    levels[4] = 1.5                                                                 # an all-equal row
    levels[9, rng.integers(0, 3000, 40)] = np.nan
    levels[11] = np.nan                                                             # nothing selectable
    levels[17, :2990] = np.nan                                                      # 10 selectable entries
    levels[20, 7] = np.inf
    levels[21, 8] = -np.inf
    spread = rng.random((5, 1500))
    return [("levels", levels), ("spread", spread)]


@pytest.mark.parametrize("k", [1, 7, 1023, 1024])
def test_row_topk_matches_the_definition_at_every_block(sb, k):
    from sympa_b200 import ops
    rng = np.random.default_rng(k)
    for name, block in synthetic_blocks(rng):
        rows, cols = block.shape
        exclude = rng.integers(-1, cols, rows)
        exclude[::3] = -1
        want = knn_oracle.topk(block, k, exclude)
        d = torch.from_numpy(block).cuda()
        ex = torch.from_numpy(exclude).cuda()
        status_bits(sb)
        assert_topk(ops.row_topk(d, k, exclude=ex), want)
        assert bool(status_bits(sb) & 8) == bool(np.isnan(block).any())
        # block heights and offsets: a row's answer does not depend on the block it comes in
        for height in (1, 3, 16):
            for r0 in range(0, rows, height * 2 + 1):
                r1 = min(rows, r0 + height)
                part = (want[0][r0:r1], want[1][r0:r1])
                assert_topk(ops.row_topk(d[r0:r1], k, exclude=ex[r0:r1]), part)
        status_bits(sb)
        # no exclusion at all
        assert_topk(ops.row_topk(d, k), knn_oracle.topk(block, k))
        status_bits(sb)


@pytest.mark.parametrize("k", [1, 7, 1023, 1024])
def test_row_topk_with_fewer_columns_than_k(sb, k):
    from sympa_b200 import ops
    rng = np.random.default_rng(3)
    for cols in (1, 5, 1000):
        if cols >= k:
            continue
        block = rng.integers(0, 3, (6, cols)).astype(np.float64)
        exclude = np.array([-1, 0, cols - 1, -1, cols // 2, 0])
        assert_topk(ops.row_topk(torch.from_numpy(block).cuda(), k, exclude=torch.from_numpy(exclude).cuda()),
                    knn_oracle.topk(block, k, exclude))


@pytest.mark.parametrize("k", [1, 7, 1023, 1024])
def test_row_topk_of_long_single_rows(sb, k):
    """2^22 columns in one row: the row is split over many CTAs and their candidates merged"""
    from sympa_b200 import ops
    rng = np.random.default_rng(40 + k)
    cols = 1 << 22
    rows = [rng.random(cols),                                                 # distinct values
            rng.integers(0, 3, cols).astype(np.float64),                      # three levels: ties decided by column
            np.full(cols, 2.0),                                               # all equal
            np.sort(rng.random(cols))[::-1].copy()]                           # descending: every tile improves
    rows[1][rng.integers(0, cols, 1000)] = np.nan
    for row in rows:
        for exclude in (-1, int(rng.integers(0, cols))):
            want = knn_oracle.topk(row[None], k, [exclude])
            got = ops.row_topk(torch.from_numpy(row[None]).cuda(), k, exclude=torch.tensor([exclude], device="cuda"))
            assert_topk(got, want)
    status_bits(sb)


def test_row_topk_bad_arguments(sb):
    import ctypes
    from sympa_b200 import _lib, ops
    d = torch.zeros(3, 10, dtype=torch.float64, device="cuda")
    for k in (0, 1025):
        with pytest.raises(ValueError):
            ops.row_topk(d, k)
    with pytest.raises(ValueError):
        ops.row_topk(d, 2, exclude=torch.zeros(2, dtype=torch.int64, device="cuda"))
    lib = _lib.load()
    assert lib.sympa_row_topk_workspace_bytes(3, 10, 0) == -1
    assert lib.sympa_row_topk_workspace_bytes(3, 10, 1025) == -1
    assert lib.sympa_row_topk_workspace_bytes(0, 10, 4) == 0
    need = lib.sympa_row_topk_workspace_bytes(3, 10, 4)
    assert need == 3 * 4 * 16                                                 # one slice per row of 10 columns
    P = ctypes.c_void_p
    out = torch.empty(3, 4, dtype=torch.int64, device="cuda")
    assert lib.sympa_row_topk(3, 10, P(d.data_ptr()), None, 4, P(out.data_ptr()), P(out.data_ptr()), P(out.data_ptr()),
                              need - 1, None, None) == 1                      # workspace too small


def manifold_and_table(sb, kind, n, metric, rows, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "spd":
        return sb.SymmetricPositiveDefinite().cuda(), so.spd_spread(rows, n, generator=g).cuda()
    table = so.upper_spread(rows, n, generator=g, scale=0.3)
    if kind == "bounded":
        table = so.to_symmetric(so.cayley_transform(table))
    cls = {"upper": sb.UpperHalfManifold, "bounded": sb.BoundedDomainManifold}[kind]
    return cls(dims=n, metric=sb.MetricType.from_str(metric)).cuda(), table.cuda()


CASES = ([(kind, n, m) for kind in ("upper", "bounded") for n in (2, 4, 7, 10) for m in METRICS]
         + [("spd", n, "riem") for n in (2, 4, 7, 10)])
ROWS = 97


def queries_for(rows):
    # scattered, repeated and the boundary ids
    return torch.tensor([5, 0, rows - 1, 41, 5, 77, 0, 13, 13, rows - 1, 64, 2], dtype=torch.int64)


@pytest.mark.parametrize("kind,n,metric", CASES)
def test_dist_rows_equal_the_rows_of_dist_matrix(sb, kind, n, metric):
    from sympa_b200 import ops
    man, t = manifold_and_table(sb, kind, n, metric, ROWS, seed=n)
    metric = "riem" if kind == "spd" else metric
    w = None if kind == "spd" else man._wsum(t)
    full = ops.dist_matrix(kind, metric, t, wsum_w=w)
    q = queries_for(ROWS).cuda()
    got = ops.dist_rows(kind, metric, t, q, w)
    assert torch.equal(bits(got), bits(full[q]))
    # small chunks: the chunk loop crosses row boundaries
    again = ops.dist_rows(kind, metric, t, q, w, chunk_pairs=1000)
    assert torch.equal(bits(again), bits(got))
    ops.check_status()


def test_dist_rows_rejects_bad_ids(sb):
    import ctypes
    from sympa_b200 import _lib, ops
    man, t = manifold_and_table(sb, "upper", 3, "riem", 20, seed=1)
    for bad in ([0, 20], [-1], [3, 5, 99]):
        with pytest.raises(ValueError, match="queries must lie"):
            ops.dist_rows("upper", "riem", t, torch.tensor(bad, device="cuda"))
    with pytest.raises(TypeError):
        ops.dist_rows("upper", "riem", t, torch.tensor([1, 2], dtype=torch.int32, device="cuda"))
    assert ops.dist_rows("upper", "riem", t, torch.empty(0, dtype=torch.int64, device="cuda")).shape == (0, 20)
    # through the C ABI, where the list is not read on the host: the row of a bad id is NaN, the status says why,
    # the other rows are untouched
    lib = _lib.load()
    q = torch.tensor([3, 20, -5, 7], dtype=torch.int64, device="cuda")
    out = torch.zeros(4, 20, dtype=torch.float64, device="cuda")
    ws = torch.empty(2 * 80, dtype=torch.int64, device="cuda")
    status_bits(sb)
    P = ctypes.c_void_p
    w = ops.status_word(t.device)
    assert lib.sympa_dist_rows(0, 3, 0, P(t.data_ptr()), 20, P(q.data_ptr()), 4, None, P(out.data_ptr()),
                               P(ws.data_ptr()), 80, P(w.data_ptr()), None) == 0
    assert torch.isnan(out[1:3]).all()
    full = ops.dist_matrix("upper", "riem", t)
    assert torch.equal(bits(out[[0, 3]]), bits(full[[3, 7]]))
    assert status_bits(sb) & 16
    assert lib.sympa_dist_rows(0, 3, 0, P(t.data_ptr()), 20, None, 4, None, P(out.data_ptr()), P(ws.data_ptr()), 80,
                               None, None) == 1


def route_matrix(sb, man, t):
    """the matrix nearest selects from: dist_matrix of the table, or for the bounded domain of its inverse Cayley
    transform (the route evaluate takes; the per-pair bounded kernels differ from it in the last bits)"""
    from sympa_b200 import metrics, ops
    src, kind, metric, wsum = metrics._distance_source(man, t)
    return ops.dist_matrix(kind, metric, src, wsum_w=wsum)


@pytest.mark.parametrize("kind,n,metric", CASES)
def test_nearest_is_the_stable_sort_of_the_matrix_rows(sb, kind, n, metric):
    from sympa_b200.metrics import nearest
    man, t = manifold_and_table(sb, kind, n, metric, ROWS, seed=n + 3)
    if kind != "bounded":
        assert torch.equal(bits(route_matrix(sb, man, t)), bits(man.dist_matrix(t)))
    d = route_matrix(sb, man, t).cpu()
    q = queries_for(ROWS)
    for k, exclude_self in ((1, True), (10, True), (ROWS - 1, True), (ROWS, False)):
        got = nearest(man, t, q.cuda(), k, exclude_self=exclude_self)
        assert got.ids.device == t.device and got.ids.shape == (q.numel(), k)
        for i, u in enumerate(q.tolist()):
            keep = torch.arange(ROWS)
            if exclude_self:
                keep = keep[keep != u]
            s = torch.sort(d[u][keep], stable=True)
            assert got.ids[i].tolist() == keep[s.indices[:k]].tolist()
            assert torch.equal(bits(got.distances[i]), bits(s.values[:k]))


def test_nearest_does_not_depend_on_blocks_or_shards(sb):
    from sympa_b200.metrics import nearest
    rows = 3000
    man, t = manifold_and_table(sb, "bounded", 4, "finf", rows, seed=8)
    rng = np.random.default_rng(8)
    q = torch.from_numpy(rng.integers(0, rows, 301)).cuda()
    one = nearest(man, t, q, 25, scale=0.7)
    d = route_matrix(sb, man, t).cpu().numpy()
    qq = q.cpu().numpy()
    want = knn_oracle.topk(d[qq], 25, qq)
    assert one.ids.cpu().tolist() == want[0].tolist()
    assert torch.equal(bits(one.distances), bits(torch.from_numpy(want[1]) * 0.7))
    for block_bytes in (8 * rows, 8 * rows * 7, 8 * rows * 300):
        again = nearest(man, t, q, 25, scale=0.7, block_bytes=block_bytes)
        assert torch.equal(again.ids, one.ids) and torch.equal(bits(again.distances), bits(one.distances))
    for world in (2, 3, 4):
        parts = [nearest(man, t, q, 25, scale=0.7, world_size=world, rank=r, block_bytes=8 * rows * 40)
                 for r in range(world)]
        assert torch.equal(torch.cat([p.ids for p in parts]), one.ids)
        assert torch.equal(bits(torch.cat([p.distances for p in parts])), bits(one.distances))


def test_nearest_of_no_queries_and_bad_arguments(sb):
    from sympa_b200 import ops
    from sympa_b200.metrics import nearest
    man, t = manifold_and_table(sb, "upper", 2, "riem", 50, seed=2)
    none = nearest(man, t, torch.empty(0, dtype=torch.int64, device="cuda"), 4)
    assert none.ids.shape == (0, 4) and none.distances.shape == (0, 4) and none.ids.is_cuda
    status_bits(sb)
    for q, k in (([0, 50], 3), ([0, 1], 50), ([0, 1], 0)):
        with pytest.raises(ValueError):
            nearest(man, t, torch.tensor(q, device="cuda"), k)
    assert status_bits(sb) == 0
    got = nearest(man, t, torch.tensor([7, 7]), 49)            # CPU queries are moved to the table's device
    assert got.ids.is_cuda and torch.equal(got.ids[0], got.ids[1]) and 7 not in got.ids[0].tolist()
    assert sorted(got.ids[0].tolist()) == [u for u in range(50) if u != 7]
    ops.check_status()


def test_nearest_memory_stays_within_the_block_and_the_outputs(sb):
    from sympa_b200 import ops
    from sympa_b200.metrics import nearest
    rows, q_count, k = 1 << 15, 3000, 100
    man, t = manifold_and_table(sb, "upper", 2, "riem", rows, seed=6)
    q = torch.from_numpy(np.random.default_rng(6).integers(0, rows, q_count)).cuda()
    block_bytes = 64 << 20
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.memory_allocated()
    got = nearest(man, t, q, k, block_bytes=block_bytes)
    growth = torch.cuda.max_memory_allocated() - before
    workspaces = sum(w.numel() * w.element_size() for cache in (ops._idx_workspace, ops._topk_workspace)
                     for w in cache.values())
    bound = block_bytes + workspaces + 16 * q_count * k + 8 * q_count + (64 << 10)
    assert growth <= bound, (growth, bound)
    assert (got.ids >= 0).all()


def test_model_nearest_uses_its_own_scale(sb):
    from sympa_b200.metrics import nearest
    from sympa_b200.model import Model
    rows = 200
    args = types.SimpleNamespace(manifold="upper", metric="riem", dims=3, num_points=rows, scale_init=1.6, scale_coef=1.0,
                                 train_scale=True)
    model = Model(args).cuda()
    model.embeddings.embeds.data.copy_(so.upper_spread(rows, 3, generator=torch.Generator().manual_seed(0)).cuda())
    q = torch.tensor([0, 199, 50, 50], dtype=torch.int64, device="cuda")
    got = model.nearest(q, 12)
    plain = nearest(model.manifold, model.embeddings.embeds, q, 12)
    scale = float(model.get_scale().detach())
    assert scale != 1.0
    assert torch.equal(got.ids, plain.ids)
    assert torch.equal(bits(got.distances), bits(plain.distances * scale))
    m = model.build_distance_matrix().cpu()
    for i, u in enumerate(q.tolist()):
        row = m[u].clone()
        row[u] = float("inf")
        s = torch.sort(row, stable=True)
        assert got.ids[i].tolist() == s.indices[:12].tolist()
        assert torch.equal(bits(got.distances[i]), bits(s.values[:12]))
