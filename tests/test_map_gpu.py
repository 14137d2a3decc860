"""Graph-reconstruction mAP on the device (sympa_average_precision, sympa_b200.metrics): the kernel on synthetic
blocks against the numpy oracle, the streaming evaluation against the oracle's own distances and bit-identical
over block sizes and row shards, bounded memory, and the reference's metric call shape."""
import ctypes
import types

import numpy as np
import pytest
import torch

import siegel_oracle as so
from map_oracle import ap_rows

pytestmark = pytest.mark.gpu

SMEM_CAP = 2048     # SY_AP_SMEM_CAP of ap_kernels.cuh: longer neighbour lists go through the workspace


@pytest.fixture(scope="module")
def sb():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    import sympa_b200
    import sympa_b200.graphs  # noqa: F401
    import sympa_b200.metrics  # noqa: F401
    from sympa_b200 import _lib
    _lib.load()
    return sympa_b200


def same_ap(a, b):
    """bit-identical per-row AP, NaN where the other has NaN"""
    a, b = a.cpu(), b.cpu()
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a[~na], b[~nb])


def close_ap(got, want, rtol=1e-14):
    got = got.cpu().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    np.testing.assert_allclose(got[ok], want[ok], rtol=rtol, atol=0)


def random_csr(sb, n, max_deg, rng, extra=None, isolated=()):
    """random graph; the nodes in `isolated` keep no edge (degree 0)"""
    src = np.repeat(np.arange(n), rng.integers(0, max_deg + 1, n))
    dst = rng.integers(0, n, src.size)
    e = torch.from_numpy(np.stack((src, dst), 1).astype(np.int64))
    if extra is not None:
        e = torch.cat((e, extra))
    if len(isolated):
        iso = torch.as_tensor(list(isolated))
        e = e[~(torch.isin(e[:, 0], iso) | torch.isin(e[:, 1], iso))]
    return sb.graphs.adjacency_csr(e, n)


def run_kernel(sb, block, row_begin, adj):
    ptr, idx = adj
    return sb.ops.average_precision(block.cuda(), row_begin, (ptr.cuda(), idx.cuda()))


# ------------------------------------------------------------------------------------------- 1. kernel
def test_kernel_random_blocks_with_offset_and_zero_degree(sb):
    rng = np.random.default_rng(1)
    n = 301
    adj = random_csr(sb, n, 6, rng, isolated=(40, 41, 60, 86))
    d = torch.from_numpy(rng.random((50, n)) * 5 + 0.01)
    deg = (adj[0][1:] - adj[0][:-1])[37:87]
    assert (deg == 0).any() and (deg > 3).any()
    ap = run_kernel(sb, d, 37, adj)
    close_ap(ap, ap_rows(d.numpy(), 37, adj[0].numpy(), adj[1].numpy()))
    sb.ops.check_status()


def test_kernel_ties(sb):
    rng = np.random.default_rng(2)
    n = 257
    adj = random_csr(sb, n, 12, rng)
    d = torch.from_numpy(rng.integers(1, 5, (n, n)).astype(np.float64))
    ap = run_kernel(sb, d, 0, adj)
    close_ap(ap, ap_rows(d.numpy(), 0, adj[0].numpy(), adj[1].numpy()))
    # the same rows in other blocks and offsets: bit-identical
    part = run_kernel(sb, d[100:107], 100, adj)
    assert same_ap(part, ap[100:107])
    sb.ops.check_status()


def test_kernel_one_row_odd_columns(sb):
    rng = np.random.default_rng(3)
    n = 999
    adj = random_csr(sb, n, 9, rng, extra=torch.tensor([[n - 1, 0], [n - 1, 5], [n - 1, 17]]))
    d = torch.from_numpy(rng.random((1, n)))
    ap = run_kernel(sb, d, n - 1, adj)
    assert ap.shape == (1,)
    close_ap(ap, ap_rows(d.numpy(), n - 1, adj[0].numpy(), adj[1].numpy()))
    sb.ops.check_status()


def test_kernel_hub_beyond_shared_memory(sb):
    rng = np.random.default_rng(4)
    n = 3 * SMEM_CAP + 11
    leaves = torch.arange(1, n)
    star = torch.stack((torch.zeros_like(leaves), leaves), 1)
    adj = random_csr(sb, n, 4, rng, extra=star)
    assert int(adj[0][1] - adj[0][0]) == n - 1 > SMEM_CAP
    d = torch.from_numpy(rng.random((5, n)) * 3)
    d[0, 1:200] = d[0, 201:400]           # ties inside the hub's list too
    ap = run_kernel(sb, d, 0, adj)
    close_ap(ap, ap_rows(d.numpy(), 0, adj[0].numpy(), adj[1].numpy()))
    sb.ops.check_status()


def test_kernel_few_rows_many_columns(sb):
    rng = np.random.default_rng(5)
    n = 1 << 20
    k = torch.arange(1, n)
    parent = torch.from_numpy((rng.random(n - 1) * np.arange(1, n)).astype(np.int64))     # random recursive tree
    hub = torch.stack((torch.full((SMEM_CAP + 500,), 1001), torch.from_numpy(rng.choice(n, SMEM_CAP + 500, replace=False))), 1)
    adj = sb.graphs.adjacency_csr(torch.cat((torch.stack((k, parent), 1), hub)), n)
    rows = 6
    assert rows < torch.cuda.get_device_properties(0).multi_processor_count
    d = torch.from_numpy(rng.random((rows, n)) + 0.5)
    ap = run_kernel(sb, d, 998, adj)
    close_ap(ap, ap_rows(d.numpy(), 998, adj[0].numpy(), adj[1].numpy()))
    sb.ops.check_status()


def test_kernel_bad_arguments_raise(sb):
    from sympa_b200 import _lib
    adj = sb.graphs.adjacency_csr(torch.tensor([[0, 1], [1, 2]]), 3)
    adj = (adj[0].cuda(), adj[1].cuda())
    d = torch.rand(2, 3, dtype=torch.float64, device="cuda")
    with pytest.raises(RuntimeError, match="no CPU path"):
        sb.ops.average_precision(d.cpu(), 0, adj)
    with pytest.raises(TypeError):
        sb.ops.average_precision(d.float(), 0, adj)
    with pytest.raises(ValueError):
        sb.ops.average_precision(d, 2, adj)                         # rows 2..3 of a 3-node graph
    with pytest.raises(ValueError):
        sb.ops.average_precision(d, 0, (adj[0][:-1], adj[1]))       # ptr of the wrong length
    with pytest.raises(ValueError):
        sb.ops.average_precision(d[0], 0, adj)
    lib = _lib.load()
    P = ctypes.c_void_p
    ws = torch.empty(64, dtype=torch.float64, device="cuda")
    # workspace: words [0, 32) of ws, ap_out: words 40, 41
    args = (P(d.data_ptr()), P(adj[0].data_ptr()), P(adj[1].data_ptr()), P(ws.data_ptr() + 8 * 40))
    assert lib.sympa_average_precision(0, 2, 3, *args, P(ws.data_ptr()), 256, None, None) == 0
    assert lib.sympa_average_precision(-1, 2, 3, *args, P(ws.data_ptr()), 256, None, None) == 1
    assert lib.sympa_average_precision(2, 2, 3, *args, P(ws.data_ptr()), 256, None, None) == 1
    assert lib.sympa_average_precision(0, 2, 3, None, *args[1:], P(ws.data_ptr()), 256, None, None) == 1
    assert lib.sympa_average_precision(0, 2, 3, *args, None, 256, None, None) == 1
    assert lib.sympa_average_precision(0, 2, 3, *args, P(ws.data_ptr()), 16, None, None) == 1     # workspace too small
    assert lib.sympa_average_precision_workspace_bytes(-1, 0) == -1
    assert lib.sympa_average_precision_workspace_bytes(3, 10) == 16 * 13
    torch.cuda.synchronize()


def test_kernel_bad_index_and_nan_set_status(sb):
    n = 6
    ptr = torch.tensor([0, 4, 6, 6, 6, 6, 6])
    idx = torch.tensor([2, n + 3, 3, -1, 0, 3])          # row 0 has two out-of-range neighbours: they are ignored
    d = torch.tensor([[0.0, 1, 2, 3, 4, 5], [1, 0.0, 2, 3, 4, 5]], dtype=torch.float64)
    sb.ops.check_status(reset=True)
    ap = sb.ops.average_precision(d.cuda(), 0, (ptr.cuda(), idx.cuda()))
    with pytest.raises(AssertionError, match="out of range"):
        sb.ops.check_status()
    # row 0: neighbours {2, 3} at 2, 3 -> 1/2, 2/3; row 1: {0, 3} at 1, 3 -> 1/1, 2/3
    assert ap[0].item() == pytest.approx((1 / 2 + 2 / 3) / 2, rel=1e-15)
    assert ap[1].item() == pytest.approx((1 + 2 / 3) / 2, rel=1e-15)
    d[1, 4] = float("nan")
    ap = sb.ops.average_precision(d.cuda(), 0, (ptr.cuda(), idx.cuda()))
    with pytest.raises(AssertionError, match="non-finite"):
        sb.ops.check_status()
    assert torch.isnan(ap[1]).item()
    sb.ops.check_status()


# ------------------------------------------------------------------------------------------- 2. streaming
def small_graph(sb, name):
    g = sb.graphs
    if name == "grid":
        ids, gd, n = g.grid_triplets(5, 2)
    elif name == "tree":
        ids, gd, n = g.balanced_tree_triplets(2, 4)
    else:
        ids, gd, n = g.product_cartesian_triplets(2, 1, 3, 2)
    return g.adjacency_csr(ids[gd == 1], n), n


def manifold_and_table(sb, kind, n, metric, rows, seed):
    g = torch.Generator().manual_seed(seed)
    w = None
    if kind == "spd":
        return sb.SymmetricPositiveDefinite().cuda(), so.spd_spread(rows, n, generator=g), None
    table = so.upper_spread(rows, n, generator=g, scale=0.3)
    if kind == "bounded":
        table = so.to_symmetric(so.cayley_transform(table))
    cls = {"upper": sb.UpperHalfManifold, "bounded": sb.BoundedDomainManifold}[kind]
    man = cls(dims=n, metric=sb.MetricType.from_str(metric)).cuda()
    if metric == "wsum":
        w = torch.linspace(0.3, 1.2, n, dtype=torch.float64).reshape(1, n)
        man.metric.weights.data = w.cuda()
    return man, table, w


def oracle_matrix(kind, metric, table, w):
    rows = table.shape[0]
    i, j = torch.meshgrid(torch.arange(rows), torch.arange(rows), indexing="ij")
    i, j = i.reshape(-1), j.reshape(-1)
    off = i != j
    d = torch.zeros(rows * rows, dtype=torch.float64)
    d[off] = so.dist(kind, table[i[off]], table[j[off]], metric, w)
    return d.reshape(rows, rows).numpy()


CASES = [("upper", 2, "riem", "grid"), ("upper", 4, "fmin", "tree"), ("upper", 7, "wsum", "product"),
         ("upper", 10, "riem", "tree"), ("bounded", 2, "fmin", "product"), ("bounded", 4, "wsum", "grid"),
         ("bounded", 7, "riem", "tree"), ("bounded", 10, "fmin", "grid"), ("spd", 3, "riem", "product"),
         ("spd", 6, "riem", "tree")]


@pytest.mark.parametrize("kind,n,metric,graph", CASES)
def test_streaming_map_matches_oracle_and_block_sizes(sb, kind, n, metric, graph):
    from sympa_b200.metrics import MeanAveragePrecisionMetric, mean_average_precision
    adj, rows = small_graph(sb, graph)
    man, table, w = manifold_and_table(sb, kind, n, metric, rows, seed=n)
    t = table.cuda()
    runs = [mean_average_precision(man, t, adj, block_bytes=8 * rows * b) for b in (1, 7, rows)]
    runs.append(mean_average_precision(man, t, adj))
    full = runs[-1][2]
    for s, c, ap in runs:
        assert same_ap(ap, full)
        assert c == rows and s == runs[-1][0]
    # the oracle on its own distances; precondition: no two distances of a row within 1e-9 relative
    dm = oracle_matrix(kind, metric, table, w)
    for u in range(rows):
        r = np.sort(np.delete(dm[u], u))
        assert np.all(np.diff(r) > 1e-9 * r[1:]), (u, np.min(np.diff(r) / r[1:]))
    close_ap(full, ap_rows(dm, 0, adj[0].numpy(), adj[1].numpy()))
    # the reference's call shape on the whole matrix: the same per-row AP (upper / spd: the same kernels wrote the
    # matrix; bounded: per-pair kernels there, the transformed table here - equal ranks by the gap precondition)
    metric_obj = MeanAveragePrecisionMetric(adj)
    mat = man.dist_matrix(t)
    assert same_ap(metric_obj.average_precision(mat), full)
    assert metric_obj.calculate_metric(mat) == pytest.approx(runs[-1][0] / rows, rel=1e-15)
    assert metric_obj.calculate_metric(mat.cpu().numpy()) == metric_obj.calculate_metric(mat)


def test_model_mean_average_precision(sb):
    from sympa_b200.metrics import mean_average_precision
    from sympa_b200.model import Model
    adj, rows = small_graph(sb, "product")
    args = types.SimpleNamespace(manifold="upper", metric="riem", dims=3, num_points=rows, scale_init=1.0, scale_coef=1.0,
                                 train_scale=False)
    model = Model(args).cuda()
    model.embeddings.embeds.data.copy_(so.upper_spread(rows, 3, generator=torch.Generator().manual_seed(0)).cuda())
    s, c, _ = mean_average_precision(model.manifold, model.embeddings.embeds, adj)
    got = model.mean_average_precision(adj, block_bytes=8 * rows * 5)
    assert isinstance(got, float) and got == s / c and 0.0 < got <= 1.0


# ------------------------------------------------------------------------------------------- 3. sharding
@pytest.mark.parametrize("world", [2, 3])
def test_row_shards_concatenate_to_the_one_rank_result(sb, world):
    from sympa_b200 import distributed as sd
    from sympa_b200.metrics import mean_average_precision
    adj, rows = small_graph(sb, "grid")
    man, table, _ = manifold_and_table(sb, "bounded", 4, "riem", rows, seed=7)
    t = table.cuda()
    _, _, one = mean_average_precision(man, t, adj, block_bytes=8 * rows * 3)
    parts = [mean_average_precision(man, t, adj, rows=sd.row_shard(rows, k, world)[:2], block_bytes=8 * rows * 3)
             for k in range(world)]
    assert same_ap(torch.cat([p[2] for p in parts]), one)
    assert sum(p[1] for p in parts) == rows


# ------------------------------------------------------------------------------------------- 4. memory
def test_memory_is_bounded_by_the_block(sb):
    from sympa_b200.metrics import mean_average_precision
    n_nodes = 1 << 15
    rng = np.random.default_rng(6)
    k = torch.arange(1, n_nodes)
    parent = torch.from_numpy((rng.random(n_nodes - 1) * np.arange(1, n_nodes)).astype(np.int64))
    adj = sb.graphs.adjacency_csr(torch.stack((k, parent), 1), n_nodes)
    man, table, _ = manifold_and_table(sb, "upper", 2, "riem", n_nodes, seed=3)
    t = table.cuda()
    adj = (adj[0].cuda(), adj[1].cuda())
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.memory_allocated()
    s, c, ap = mean_average_precision(man, t, adj, block_bytes=64 << 20)
    growth = torch.cuda.max_memory_allocated() - before
    assert growth < (1 << 29), growth          # the whole matrix would be 8.6 GB
    assert c == n_nodes and 0.0 < s / c <= 1.0
    _, _, spot = mean_average_precision(man, t, adj, rows=(20000, 20600), block_bytes=1 << 30)
    assert same_ap(spot, ap[20000:20600])
