"""Graph-reconstruction distortion on the device (sympa_hop_distances, sympa_distortion_rows, sympa_b200.metrics):
hop distances against scipy's csgraph on awkward graphs and at every block shape, the triplets built from them
against the closed-form generators, the distortion kernel against the numpy oracle, the streaming evaluation
against the reference's route over triplets, bit-identical over block sizes and row shards, one pass shared with
mAP, bounded memory and the model's own scale."""
import ctypes
import types

import numpy as np
import pytest
import torch

import siegel_oracle as so
from distortion_oracle import distortion, distortion_rows, hop_matrix

pytestmark = pytest.mark.gpu

# SY_HOP_SMEM_VISITED_BYTES of hop_kernels.cuh, in bits: larger graphs keep the BFS visited set in global memory
SMEM_VISITED_NODES = (48 * 1024 - 256) * 8


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


def csr(sb, edges, n):
    ptr, idx = sb.graphs.adjacency_csr(torch.as_tensor(edges, dtype=torch.int64).reshape(-1, 2), n)
    return ptr, idx


def random_components(sb, rng):
    """three random graphs on disjoint node ranges plus isolated nodes"""
    parts, n = [], 0
    for size, deg in ((300, 2), (150, 1), (90, 4)):
        src = np.repeat(np.arange(size), rng.integers(0, deg + 1, size))
        parts.append(np.stack((src, rng.integers(0, size, src.size)), 1) + n)
        n += size
    n += 17                                   # nodes 540..556 have no edge
    e = np.concatenate(parts)
    return csr(sb, e, n), n


def random_tree(rng, n):
    k = np.arange(1, n)
    return np.stack((k, (rng.random(n - 1) * k).astype(np.int64)), 1)      # parent of k drawn from [0, k)


def hop_blocks(sb, adj, begin, end, height):
    """rows [begin, end) of the hop matrix through ops.hop_distances in blocks of `height` rows"""
    dev = (adj[0].cuda(), adj[1].cuda())
    return torch.cat([sb.ops.hop_distances(dev, r0, min(height, end - r0)) for r0 in range(begin, end, height)]).cpu()


# ------------------------------------------------------------------------------------------- 1. hop distances
def graph_case(sb, name):
    rng = np.random.default_rng(11)
    if name == "components":
        return random_components(sb, rng)
    if name == "path":
        n = 3000
        perm = rng.permutation(n)                  # a path whose node ids are shuffled
        return csr(sb, np.stack((perm[:-1], perm[1:]), 1), n), n
    if name == "star":
        n = 3 * 2048 + 11                          # the hub's list is longer than any shared-memory cap
        leaves = np.arange(1, n)
        e = np.concatenate((np.stack((np.zeros_like(leaves), leaves), 1), random_tree(rng, n)[::7]))
        return csr(sb, e, n), n
    ids, gd, n = sb.graphs.grid_triplets(20, 2)
    return sb.graphs.adjacency_csr(ids[gd == 1], n), n


@pytest.mark.parametrize("name", ["components", "path", "star", "grid"])
def test_hop_distances_match_scipy_at_every_block_shape(sb, name):
    adj, n = graph_case(sb, name)
    want = hop_matrix(adj[0].numpy(), adj[1].numpy())
    sb.ops.check_status(reset=True)
    full = hop_blocks(sb, adj, 0, n, n)
    assert full.dtype == torch.int32 and full.shape == (n, n)
    np.testing.assert_array_equal(full.numpy(), want)
    for height in (1, 7, 128):
        for begin in (0, 5, n // 2 + 3):
            end = min(n, begin + 3 * height + 2)
            assert torch.equal(hop_blocks(sb, adj, begin, end, height), full[begin:end]), (height, begin)
    if name == "components":
        assert (full == -1).any() and (full[545] == -1).sum() == n - 1
    sb.ops.check_status()


def test_hop_distances_rows_of_a_random_tree_of_2_20_nodes(sb):
    rng = np.random.default_rng(12)
    n = 1 << 20
    adj = csr(sb, random_tree(rng, n), n)
    rows = np.arange(998, 1004)
    want = hop_matrix(adj[0].numpy(), adj[1].numpy(), rows=rows)
    got = hop_blocks(sb, adj, 998, 1004, 6)
    np.testing.assert_array_equal(got.numpy(), want)
    assert torch.equal(hop_blocks(sb, adj, 998, 1004, 1), got)
    assert torch.equal(hop_blocks(sb, adj, 998, 1004, 4), got)
    sb.ops.check_status()


@pytest.mark.parametrize("n", [SMEM_VISITED_NODES, SMEM_VISITED_NODES + 1, 393216])
def test_hop_distances_at_the_shared_memory_boundary(sb, n):
    """the largest graph with the visited bitmap in shared memory, the smallest without, and 48 KB of bits"""
    rng = np.random.default_rng(15)
    adj = csr(sb, random_tree(rng, n), n)
    rows = np.r_[0:3, n - 4:n]
    want = hop_matrix(adj[0].numpy(), adj[1].numpy(), rows=rows)
    sb.ops.check_status(reset=True)
    got = torch.cat((hop_blocks(sb, adj, 0, 3, 3), hop_blocks(sb, adj, n - 4, n, 2)))
    np.testing.assert_array_equal(got.numpy(), want)
    sb.ops.check_status()


def test_hop_distances_bad_index_on_the_global_path(sb):
    n = SMEM_VISITED_NODES + 1
    rng = np.random.default_rng(16)
    ptr, idx = csr(sb, random_tree(rng, n), n)
    rows = np.arange(n - 3, n)
    want = hop_matrix(ptr.numpy(), idx.numpy(), rows=rows)
    # two out-of-range entries appended to the last node's list: skipped, every distance unchanged
    idx = torch.cat((idx, torch.tensor([n + 7, -3])))
    ptr = ptr.clone()
    ptr[-1] += 2
    sb.ops.check_status(reset=True)
    got = sb.ops.hop_distances((ptr.cuda(), idx.cuda()), n - 3, 3)
    with pytest.raises(AssertionError, match="out of range"):
        sb.ops.check_status()
    np.testing.assert_array_equal(got.cpu().numpy(), want)


def test_hop_distances_bad_index_sets_status(sb):
    n = 5
    ptr = torch.tensor([0, 3, 4, 5, 5, 5]).cuda()
    idx = torch.tensor([1, n + 2, -4, 0, 0]).cuda()        # row 0 has two out-of-range entries: skipped
    sb.ops.check_status(reset=True)
    h = sb.ops.hop_distances((ptr, idx), 0, n)
    with pytest.raises(AssertionError, match="out of range"):
        sb.ops.check_status()
    # directed as stored: 0 -> 1, 1 -> 0, 2 -> 0
    assert h.cpu().tolist()[0] == [0, 1, -1, -1, -1]
    assert h.cpu().tolist()[2] == [1, 2, 0, -1, -1]


def test_hop_distances_bad_arguments(sb):
    from sympa_b200 import _lib
    lib = _lib.load()
    adj = csr(sb, [[0, 1], [1, 2]], 3)
    ptr, idx = adj[0].cuda(), adj[1].cuda()
    with pytest.raises(RuntimeError, match="no CPU path"):
        sb.ops.hop_distances(adj, 0, 3)
    with pytest.raises(ValueError):
        sb.ops.hop_distances((ptr, idx), 2, 2)
    with pytest.raises(ValueError):
        sb.ops.hop_distances((ptr, idx), 0, 3, out=torch.empty(3, 3, dtype=torch.int64, device="cuda"))
    P = ctypes.c_void_p
    nbytes = lib.sympa_hop_distances_workspace_bytes(3)
    assert nbytes >= 256 + 3 * 4 and lib.sympa_hop_distances_workspace_bytes(-1) == -1
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    out = torch.empty(3, 3, dtype=torch.int32, device="cuda")
    args = (P(ptr.data_ptr()), P(idx.data_ptr()), P(out.data_ptr()), P(ws.data_ptr()))
    assert lib.sympa_hop_distances(0, 3, 3, *args, nbytes, None, None) == 0
    assert lib.sympa_hop_distances(-1, 2, 3, *args, nbytes, None, None) == 1
    assert lib.sympa_hop_distances(0, -1, 3, *args, nbytes, None, None) == 1
    assert lib.sympa_hop_distances(2, 2, 3, *args, nbytes, None, None) == 1          # rows 2..3 of 3 nodes
    assert lib.sympa_hop_distances(0, 3, 3, *args, nbytes - 1, None, None) == 1      # workspace too small
    assert lib.sympa_hop_distances(0, 3, 3, *args[:3], None, nbytes, None, None) == 1
    torch.cuda.synchronize()
    assert out.cpu().tolist() == [[0, 1, 2], [1, 0, 1], [2, 1, 0]]


# ------------------------------------------------------------------------------------------- 2. triplets
@pytest.mark.parametrize("gen,args", [("grid_triplets", (5, 2)), ("balanced_tree_triplets", (2, 4)),
                                      ("product_cartesian_triplets", (2, 1, 3, 2))])
def test_shortest_path_triplets_equal_the_generators(sb, gen, args):
    ids, gd, n = getattr(sb.graphs, gen)(*args)
    adj = sb.graphs.adjacency_csr(ids[gd == 1], n)
    for block_bytes in (4 * n * 3, 1 << 30):
        got_ids, got_d, got_n = sb.graphs.shortest_path_triplets(adj, block_bytes=block_bytes)
        assert got_n == n and got_ids.device == ids.device and got_d.dtype == torch.float64
        assert torch.equal(got_ids, ids) and torch.equal(got_d, gd)
    cuda_ids, cuda_d, _ = sb.graphs.shortest_path_triplets((adj[0].cuda(), adj[1].cuda()))
    assert cuda_ids.is_cuda and torch.equal(cuda_ids.cpu(), ids) and torch.equal(cuda_d.cpu(), gd)


def test_shortest_path_triplets_skip_unconnected_pairs(sb):
    adj = csr(sb, [[0, 1], [1, 2], [3, 4]], 6)
    ids, d, n = sb.graphs.shortest_path_triplets(adj)
    assert n == 6 and ids.tolist() == [[0, 1], [0, 2], [1, 2], [3, 4]] and d.tolist() == [1.0, 2.0, 1.0, 1.0]


# ------------------------------------------------------------------------------------------- 3. distortion kernel
def close_rows(got, want, rtol=1e-14):
    s, c, hi, lo = (t.cpu().numpy() for t in got)
    np.testing.assert_array_equal(c, want[1])
    for g, w in ((s, want[0]), (hi, want[2]), (lo, want[3])):
        ok = np.isfinite(w)
        np.testing.assert_array_equal(g[~ok], w[~ok])          # NaN and +-inf in the same places
        np.testing.assert_allclose(g[ok], w[ok], rtol=rtol, atol=0)


def same_rows(a, b):
    """bit-identical DistortionRows, NaN where the other has NaN"""
    for x, y in zip(a, b):
        x, y = x.cpu(), y.cpu()
        if x.dtype.is_floating_point:
            nx_, ny_ = torch.isnan(x), torch.isnan(y)
            if not (torch.equal(nx_, ny_) and torch.equal(x[~nx_], y[~ny_])):
                return False
        elif not torch.equal(x, y):
            return False
    return True


def test_distortion_rows_match_the_oracle(sb):
    rng = np.random.default_rng(13)
    adj, n = random_components(sb, rng)
    begin, rows = 37, 120
    h = hop_matrix(adj[0].numpy(), adj[1].numpy(), rows=np.arange(begin, begin + rows))
    d = rng.random((rows, n)) * 4 + 0.01
    assert (h == -1).any()
    for scale in (1.0, 0.37):
        got = sb.ops.distortion_rows(torch.from_numpy(d).cuda(), torch.from_numpy(h).cuda(), begin, scale)
        close_rows(got, distortion_rows(d, h, begin, scale))
    # other blocks and offsets holding the same rows: bit-identical
    full = sb.ops.distortion_rows(torch.from_numpy(d).cuda(), torch.from_numpy(h).cuda(), begin, 0.37)
    part = sb.ops.distortion_rows(torch.from_numpy(d[40:47]).cuda(), torch.from_numpy(h[40:47]).cuda(), begin + 40, 0.37)
    assert same_rows(part, tuple(t[40:47] for t in full))
    sb.ops.check_status()


def test_distortion_rows_nan_row_sets_status(sb):
    rng = np.random.default_rng(14)
    n = 64
    adj = csr(sb, random_tree(rng, n), n)
    h = hop_matrix(adj[0].numpy(), adj[1].numpy())
    d = rng.random((n, n)) + 0.5
    d[3, 40] = np.nan                               # row 3 (a pair 3 < 40): NaN terms
    d[50, 10] = np.nan                              # row 50, column 10 < 50: not one of its pairs
    sb.ops.check_status(reset=True)
    got = sb.ops.distortion_rows(torch.from_numpy(d).cuda(), torch.from_numpy(h).cuda(), 0, 1.5)
    with pytest.raises(AssertionError, match="non-finite"):
        sb.ops.check_status()
    want = distortion_rows(d, h, 0, 1.5)
    close_rows(got, want)
    assert torch.isnan(got.sum[3]) and torch.isnan(got.max[3]) and torch.isnan(got.min[3])
    assert not torch.isnan(got.sum[50]) and got.count[n - 1] == 0 and got.max[n - 1] == -np.inf
    sb.ops.check_status()


def test_distortion_rows_bad_arguments(sb):
    from sympa_b200 import _lib
    lib = _lib.load()
    d = torch.rand(2, 3, dtype=torch.float64, device="cuda")
    h = torch.ones(2, 3, dtype=torch.int32, device="cuda")
    with pytest.raises(RuntimeError, match="no CPU path"):
        sb.ops.distortion_rows(d.cpu(), h, 0, 1.0)
    with pytest.raises(TypeError):
        sb.ops.distortion_rows(d, h.long(), 0, 1.0)
    with pytest.raises(ValueError):
        sb.ops.distortion_rows(d, h, 2, 1.0)
    with pytest.raises(ValueError):
        sb.ops.distortion_rows(d, h[:1], 0, 1.0)
    P = ctypes.c_void_p
    o = torch.empty(4, 2, dtype=torch.float64, device="cuda")
    outs = tuple(P(o[k].data_ptr()) for k in range(4))
    assert lib.sympa_distortion_rows(0, 2, 3, P(d.data_ptr()), P(h.data_ptr()), 1.0, *outs, None, None) == 0
    assert lib.sympa_distortion_rows(-1, 2, 3, P(d.data_ptr()), P(h.data_ptr()), 1.0, *outs, None, None) == 1
    assert lib.sympa_distortion_rows(0, -2, 3, P(d.data_ptr()), P(h.data_ptr()), 1.0, *outs, None, None) == 1
    assert lib.sympa_distortion_rows(2, 2, 3, P(d.data_ptr()), P(h.data_ptr()), 1.0, *outs, None, None) == 1
    assert lib.sympa_distortion_rows(0, 2, 3, None, P(h.data_ptr()), 1.0, *outs, None, None) == 1
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------- 4. streaming
def manifold_and_table(sb, kind, n, metric, rows, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "spd":
        return sb.SymmetricPositiveDefinite().cuda(), so.spd_spread(rows, n, generator=g)
    table = so.upper_spread(rows, n, generator=g, scale=0.3)
    if kind == "bounded":
        table = so.to_symmetric(so.cayley_transform(table))
    cls = {"upper": sb.UpperHalfManifold, "bounded": sb.BoundedDomainManifold}[kind]
    man = cls(dims=n, metric=sb.MetricType.from_str(metric)).cuda()
    if metric == "wsum":
        man.metric.weights.data = torch.linspace(0.3, 1.2, n, dtype=torch.float64).reshape(1, n).cuda()
    return man, table


def product_graph(sb):
    ids, gd, n = sb.graphs.product_cartesian_triplets(2, 1, 3, 2)
    return ids, gd, sb.graphs.adjacency_csr(ids[gd == 1], n), n


CASES = [("upper", 2, "riem"), ("upper", 4, "fmin"), ("upper", 7, "wsum"), ("upper", 10, "riem"),
         ("bounded", 2, "fone"), ("bounded", 4, "riem"), ("bounded", 7, "finf"), ("bounded", 10, "fmin"),
         ("spd", 3, "riem"), ("spd", 6, "riem")]


@pytest.mark.parametrize("kind,n,metric", CASES)
def test_average_distortion_matches_the_triplet_route(sb, kind, n, metric):
    from sympa_b200.metrics import average_distortion, worst_case
    ids, gd, adj, rows = product_graph(sb)
    man, table = manifold_and_table(sb, kind, n, metric, rows, seed=n)
    t = table.cuda()
    scale = 0.73
    total, count, hi, lo, per_row = average_distortion(man, t, adj, scale=scale)
    # the reference's route: model(triplets) = dist_from_table(table, ids) * scale, then the formula
    with torch.no_grad():
        sd = (man.dist_from_table(t, ids.cuda()) * scale).cpu().numpy()
    avg, worst = distortion(sd, gd.numpy())
    assert count == ids.shape[0]
    assert total / count == pytest.approx(avg, rel=1e-12, abs=0)
    assert worst_case(hi, lo) == pytest.approx(worst, rel=1e-12, abs=0)
    assert per_row.count.sum().item() == count and per_row.sum.shape == (rows,)
    # bit-identical per row over block sizes (1, 7 and all rows per block)
    for b in (1, 7):
        again = average_distortion(man, t, adj, scale=scale, block_bytes=12 * rows * b)
        assert same_rows(again[4], per_row) and again[:4] == (total, count, hi, lo)


@pytest.mark.parametrize("world", [2, 3])
def test_row_shards_concatenate_to_the_one_rank_result(sb, world):
    from sympa_b200 import distributed as sd
    from sympa_b200.metrics import average_distortion
    _, _, adj, rows = product_graph(sb)
    man, table = manifold_and_table(sb, "bounded", 4, "riem", rows, seed=7)
    t = table.cuda()
    one = average_distortion(man, t, adj, scale=1.3, block_bytes=12 * rows * 3)
    parts = [average_distortion(man, t, adj, scale=1.3, rows=sd.row_shard(rows, k, world)[:2], block_bytes=12 * rows * 2)
             for k in range(world)]
    assert same_rows(tuple(torch.cat([p[4][f] for p in parts]) for f in range(4)), one[4])
    assert sum(p[1] for p in parts) == one[1]
    assert max(p[2] for p in parts) == one[2] and min(p[3] for p in parts) == one[3]


def test_evaluate_is_bit_identical_to_the_separate_metrics(sb):
    from sympa_b200.metrics import average_distortion, evaluate, mean_average_precision, worst_case
    _, _, adj, rows = product_graph(sb)
    man, table = manifold_and_table(sb, "upper", 6, "finf", rows, seed=5)
    t = table.cuda()
    s_ap, c_ap, ap = mean_average_precision(man, t, adj)
    total, count, hi, lo, per_row = average_distortion(man, t, adj, scale=2.5)
    for block_bytes in (12 * rows * 4, 1 << 30):
        r = evaluate(man, t, adj, scale=2.5, block_bytes=block_bytes)
        assert r.mean_ap == s_ap / c_ap
        assert torch.equal(torch.isnan(r.ap), torch.isnan(ap)) and torch.equal(r.ap[~torch.isnan(ap)], ap[~torch.isnan(ap)])
        assert r.average_distortion == total / count and r.worst_case_distortion == worst_case(hi, lo)
        assert same_rows(r.distortion, per_row)


# ------------------------------------------------------------------------------------------- 5. memory
def test_memory_is_bounded_by_the_block(sb):
    from sympa_b200 import ops
    from sympa_b200.metrics import evaluate
    n_nodes = 1 << 15
    rng = np.random.default_rng(6)
    adj = csr(sb, random_tree(rng, n_nodes), n_nodes)
    adj = (adj[0].cuda(), adj[1].cuda())
    man, table = manifold_and_table(sb, "upper", 2, "riem", n_nodes, seed=3)
    t = table.cuda()
    block_bytes = 64 << 20
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.memory_allocated()
    r = evaluate(man, t, adj, scale=1.7, block_bytes=block_bytes)
    growth = torch.cuda.max_memory_allocated() - before
    # the kernels' workspaces (kept per device, allocated by the first call that needs them)
    workspaces = sum(w.numel() * w.element_size() for cache in (ops._hop_workspace, ops._ap_workspace, ops._idx_workspace)
                     for w in cache.values())
    assert growth <= block_bytes + workspaces + 128 * n_nodes, (growth, workspaces)
    assert growth < (1 << 30)                  # the whole matrix would be 8.6 GB of distances + 4.3 GB of hops
    assert r.distortion.count.sum().item() == n_nodes * (n_nodes - 1) // 2      # a tree is connected
    spot = evaluate(man, t, adj, scale=1.7, rows=(20000, 20600))
    assert same_rows(spot.distortion, tuple(x[20000:20600] for x in r.distortion))


# ------------------------------------------------------------------------------------------- 6. model
def test_model_evaluate_uses_its_own_scale(sb):
    from sympa_b200.metrics import mean_average_precision
    from sympa_b200.model import Model
    ids, gd, adj, rows = product_graph(sb)
    args = types.SimpleNamespace(manifold="upper", metric="riem", dims=3, num_points=rows, scale_init=1.6, scale_coef=1.0,
                                 train_scale=True)
    model = Model(args).cuda()
    model.embeddings.embeds.data.copy_(so.upper_spread(rows, 3, generator=torch.Generator().manual_seed(0)).cuda())
    with torch.no_grad():
        sd = model(ids.cuda()).cpu().numpy()                # the reference's evaluate: model(triplets)
    avg, _ = distortion(sd, gd.numpy())
    got_avg, got_map = model.evaluate(adj, block_bytes=12 * rows * 5)
    assert got_avg == pytest.approx(avg, rel=1e-12, abs=0)
    assert model.average_distortion(adj) == got_avg
    s, c, _ = mean_average_precision(model.manifold, model.embeddings.embeds, adj)
    assert got_map == s / c == model.mean_average_precision(adj)
