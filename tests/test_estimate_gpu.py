"""Sampled-row estimates on the device (sympa_distortion_rows_full, sympa_b200.metrics.estimate): the whole-row
distortion kernel against an all-columns oracle at every block shape, estimate at S = N against evaluate, a sampled
node's AP bit-identical to evaluate's, invariance to the block size and the row shards, the coverage of the
standard errors on a random tree, bounded memory and the model's own scale."""
import types

import numpy as np
import pytest
import torch

import siegel_oracle as so
from distortion_oracle import hop_matrix

pytestmark = pytest.mark.gpu


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
    return sb.graphs.adjacency_csr(torch.as_tensor(edges, dtype=torch.int64).reshape(-1, 2), n)


def random_tree(rng, n):
    k = np.arange(1, n)
    return np.stack((k, (rng.random(n - 1) * k).astype(np.int64)), 1)


def random_components(sb, rng):
    """three random graphs on disjoint node ranges plus isolated nodes"""
    parts, n = [], 0
    for size, deg in ((300, 2), (150, 1), (90, 4)):
        src = np.repeat(np.arange(size), rng.integers(0, deg + 1, size))
        parts.append(np.stack((src, rng.integers(0, size, src.size)), 1) + n)
        n += size
    n += 17
    return csr(sb, np.concatenate(parts), n), n


def full_rows_oracle(d, h, nodes, scale):
    """per row r, node u = nodes[r]: over every column w != u with h >= 1, (sum of |s d - g| / g, count, max s d / g,
    min s d / g); a NaN scaled distance among them makes the three floats NaN"""
    rows = d.shape[0]
    out = (np.zeros(rows), np.zeros(rows, dtype=np.int64), np.full(rows, -np.inf), np.full(rows, np.inf))
    for r in range(rows):
        cols = np.flatnonzero(h[r] >= 1)
        cols = cols[cols != nodes[r]]
        out[1][r] = cols.size
        if cols.size == 0:
            continue
        sd, g = scale * d[r, cols], h[r, cols].astype(np.float64)
        if np.isnan(sd).any():
            out[0][r] = out[2][r] = out[3][r] = np.nan
            continue
        out[0][r] = (np.abs(sd - g) / g).sum()
        out[2][r], out[3][r] = (sd / g).max(), (sd / g).min()
    return out


def close_rows(got, want, rtol=1e-14):
    s, c, hi, lo = (t.cpu().numpy() for t in got)
    np.testing.assert_array_equal(c, want[1])
    for g, w in ((s, want[0]), (hi, want[2]), (lo, want[3])):
        ok = np.isfinite(w)
        np.testing.assert_array_equal(g[~ok], w[~ok])
        np.testing.assert_allclose(g[ok], w[ok], rtol=rtol, atol=0)


def same(a, b):
    """bit-identical tensors, NaN where the other has NaN"""
    a, b = a.cpu(), b.cpu()
    if a.dtype.is_floating_point:
        na, nb = torch.isnan(a), torch.isnan(b)
        return torch.equal(na, nb) and torch.equal(a[~na], b[~nb])
    return torch.equal(a, b)


def same_rows(a, b):
    return all(same(x, y) for x, y in zip(a, b))


# ------------------------------------------------------------------------------------------- 1. whole-row kernel
def test_distortion_rows_full_match_the_oracle_at_every_block(sb):
    rng = np.random.default_rng(21)
    adj, n = random_components(sb, rng)
    h = hop_matrix(adj[0].numpy(), adj[1].numpy())
    d = rng.random((n, n)) * 4 + 0.01
    u = next(v for v in range(1, n) if (h[v, :v] >= 1).any())
    d[u, np.flatnonzero(h[u, :u] >= 1)[0]] = np.nan     # below the diagonal: still one of row u's whole-row pairs
    assert h[77, 500] == -1
    d[77, 500] = np.nan                                 # another component: not a pair
    h_c, d_c = torch.from_numpy(h).cuda(), torch.from_numpy(d).cuda()
    sb.ops.check_status(reset=True)
    full = sb.ops.distortion_rows(d_c, h_c, 0, 0.37, full=True)
    with pytest.raises(AssertionError, match="non-finite"):
        sb.ops.check_status()
    want = full_rows_oracle(d, h, np.arange(n), 0.37)
    close_rows(full, want)
    assert torch.isnan(full.sum[u]) and not torch.isnan(full.sum[77])
    assert (full.count.cpu().numpy() == (h >= 1).sum(1)).all() and full.count[n - 1] == 0 and full.max[n - 1] == -np.inf
    # the upper-part kernel is unchanged; the whole row holds both orders of each pair
    upper = sb.ops.distortion_rows(d_c, h_c, 0, 0.37)
    assert upper.count.sum().item() * 2 == full.count.sum().item()
    # every block height and offset: bit-identical to the one-block values
    for height in (1, 2, 7, 64, 255, 256, 257):
        for begin in (0, 3, 130):
            end = min(n, begin + 2 * height + 1)
            parts = [sb.ops.distortion_rows(d_c[r0:min(end, r0 + height)], h_c[r0:min(end, r0 + height)], r0, 0.37,
                                            full=True) for r0 in range(begin, end, height)]
            got = tuple(torch.cat([p[f] for p in parts]) for f in range(4))
            assert same_rows(got, tuple(t[begin:end] for t in full)), (height, begin)
    assert u < 515
    with pytest.raises(AssertionError, match="non-finite"):     # row u again, in the blocks that held it
        sb.ops.check_status()
    for scale in (1.0, 2.5):
        close_rows(sb.ops.distortion_rows(d_c[40:47], h_c[40:47], 40, scale, full=True),
                   full_rows_oracle(d[40:47], h[40:47], np.arange(40, 47), scale))
    sb.ops.check_status()


def test_distortion_rows_full_bad_arguments(sb):
    import ctypes
    from sympa_b200 import _lib
    lib = _lib.load()
    d = torch.rand(2, 3, dtype=torch.float64, device="cuda")
    h = torch.ones(2, 3, dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError):
        sb.ops.distortion_rows(d, h, 2, 1.0, full=True)
    P = ctypes.c_void_p
    o = torch.empty(4, 2, dtype=torch.float64, device="cuda")
    outs = tuple(P(o[k].data_ptr()) for k in range(4))
    f = lib.sympa_distortion_rows_full
    assert f(0, 2, 3, P(d.data_ptr()), P(h.data_ptr()), 1.0, *outs, None, None) == 0
    assert f(-1, 2, 3, P(d.data_ptr()), P(h.data_ptr()), 1.0, *outs, None, None) == 1
    assert f(2, 2, 3, P(d.data_ptr()), P(h.data_ptr()), 1.0, *outs, None, None) == 1
    assert f(0, 2, 3, None, P(h.data_ptr()), 1.0, *outs, None, None) == 1
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------- 2. estimate
def manifold_and_table(sb, kind, n, metric, rows, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "spd":
        return sb.SymmetricPositiveDefinite().cuda(), so.spd_spread(rows, n, generator=g)
    table = so.upper_spread(rows, n, generator=g, scale=0.3)
    if kind == "bounded":
        table = so.to_symmetric(so.cayley_transform(table))
    cls = {"upper": sb.UpperHalfManifold, "bounded": sb.BoundedDomainManifold}[kind]
    return cls(dims=n, metric=sb.MetricType.from_str(metric)).cuda(), table


def product_graph(sb):
    ids, gd, n = sb.graphs.product_cartesian_triplets(2, 2, 4, 2)         # 112 nodes
    return sb.graphs.adjacency_csr(ids[gd == 1], n), n


CASES = [("upper", 2, "riem"), ("upper", 4, "fmin"), ("upper", 7, "finf"), ("upper", 10, "riem"),
         ("bounded", 2, "fone"), ("bounded", 4, "riem"), ("bounded", 7, "finf"), ("bounded", 10, "fmin"),
         ("spd", 3, "riem")]


@pytest.mark.parametrize("kind,n,metric", CASES)
def test_estimate_of_every_row_equals_evaluate(sb, kind, n, metric):
    from sympa_b200.metrics import estimate, evaluate
    adj, rows = product_graph(sb)
    man, table = manifold_and_table(sb, kind, n, metric, rows, seed=n + 1)
    t = table.cuda()
    exact = evaluate(man, t, adj, scale=0.81)
    est = estimate(man, t, adj, rows, scale=0.81, seed=3)
    assert est.mean_ap_se == 0.0 and est.average_distortion_se == 0.0
    assert est.mean_ap == pytest.approx(exact.mean_ap, rel=1e-12, abs=0)
    assert est.average_distortion == pytest.approx(exact.average_distortion, rel=1e-12, abs=0)
    assert est.sampled_worst_case_distortion == pytest.approx(exact.worst_case_distortion, rel=1e-12, abs=0)
    assert sorted(est.nodes.tolist()) == list(range(rows))
    assert same(est.ap, exact.ap[est.nodes])
    # whole rows: every connected pair twice
    assert est.distortion.count.sum().item() == 2 * exact.distortion.count.sum().item()


def test_sampled_ap_is_bit_identical_and_block_size_does_not_matter(sb):
    from sympa_b200.metrics import estimate, evaluate, sample_order
    rng = np.random.default_rng(22)
    adj, n = random_components(sb, rng)
    man, table = manifold_and_table(sb, "bounded", 4, "riem", n, seed=2)
    t = table.cuda()
    exact = evaluate(man, t, adj, scale=1.3)
    est = estimate(man, t, adj, 100, scale=1.3, seed=9, epoch=4)
    assert est.nodes.tolist() == sample_order(n, 100, seed=9, epoch=4)[:100].tolist()
    assert same(est.ap, exact.ap[est.nodes]) and torch.isnan(est.ap).any()       # isolated nodes sampled too
    # the whole-row terms of a sampled node, against the oracle on its own rows of the exact matrices
    d = man.dist_matrix(t).cpu().numpy()
    h = hop_matrix(adj[0].numpy(), adj[1].numpy())
    rows = est.nodes.cpu().numpy()
    close_rows(est.distortion, full_rows_oracle(d[rows], h[rows], rows, 1.3), rtol=1e-13)
    for block_bytes in (12 * n, 12 * n * 7, 1 << 30):
        again = estimate(man, t, adj, 100, scale=1.3, seed=9, epoch=4, block_bytes=block_bytes)
        assert same(again.ap, est.ap) and same_rows(again.distortion, est.distortion)
        assert again[:5] == est[:5]


@pytest.mark.parametrize("world", [2, 3])
def test_rank_shards_concatenate_to_the_one_rank_values(sb, world, monkeypatch):
    """each rank's part run in one process (the all-reduces made no-ops): the per-node values concatenate to the
    one-rank result bit for bit"""
    import torch.distributed as dist
    from sympa_b200.metrics import estimate
    adj, rows = product_graph(sb)
    man, table = manifold_and_table(sb, "upper", 6, "finf", rows, seed=4)
    t = table.cuda()
    one = estimate(man, t, adj, 77, scale=0.6, seed=1, block_bytes=12 * rows * 5)
    monkeypatch.setattr(dist, "all_reduce", lambda tensor, op=None: None)
    parts = [estimate(man, t, adj, 77, scale=0.6, seed=1, block_bytes=12 * rows * 3, world_size=world, rank=k)
             for k in range(world)]
    assert same(torch.cat([p.nodes for p in parts]), one.nodes)
    assert same(torch.cat([p.ap for p in parts]), one.ap)
    assert same_rows(tuple(torch.cat([p.distortion[f] for p in parts]) for f in range(4)), one.distortion)


def walk_table(parent, n, seed):
    """upper half-space points X + i I whose X is the parent's plus a random symmetric step: neighbours lie close,
    as in a trained embedding (with independent random points AP is about 1 / uniform rank, too heavy-tailed for a
    sample of hundreds to show its spread)"""
    rng = np.random.default_rng(seed)
    steps = rng.normal(0.0, 0.3, (parent.size + 1, n, n))
    steps = 0.5 * (steps + steps.transpose(0, 2, 1))
    x = steps.copy()
    for k in range(1, parent.size + 1):
        x[k] = x[parent[k - 1]] + steps[k]
    y = np.broadcast_to(np.eye(n), x.shape)
    return so.cplx(torch.from_numpy(x), torch.from_numpy(y.copy()))


def test_standard_errors_cover_the_exact_values(sb):
    """2^14-node random tree, 20 fixed seeds at S = 512: the exact value lies within 3 standard errors of the
    estimate for at least 18 of them, for both metrics (the seeds are fixed, so the outcome is deterministic)"""
    from sympa_b200.metrics import estimate, evaluate
    n = 1 << 14
    rng = np.random.default_rng(23)
    edges = random_tree(rng, n)
    adj = csr(sb, edges, n)
    adj = (adj[0].cuda(), adj[1].cuda())
    man = sb.UpperHalfManifold(dims=2, metric=sb.MetricType.from_str("riem")).cuda()
    t = walk_table(edges[:, 1], 2, seed=5).cuda()
    exact = evaluate(man, t, adj, scale=2.0)
    z_ap, z_d = [], []
    for seed in range(20):
        est = estimate(man, t, adj, 512, scale=2.0, seed=seed)
        assert est.mean_ap_se > 0 and est.average_distortion_se > 0
        assert est.sampled_worst_case_distortion <= exact.worst_case_distortion * (1 + 1e-12)      # a lower bound
        z_ap.append(abs(est.mean_ap - exact.mean_ap) / est.mean_ap_se)
        z_d.append(abs(est.average_distortion - exact.average_distortion) / est.average_distortion_se)
    assert sum(z <= 3 for z in z_ap) >= 18 and sum(z <= 3 for z in z_d) >= 18, (z_ap, z_d)


def test_memory_stays_within_the_stated_bound(sb):
    from sympa_b200 import ops
    from sympa_b200.metrics import estimate
    n = 1 << 15
    rng = np.random.default_rng(24)
    adj = csr(sb, random_tree(rng, n), n)
    adj = (adj[0].cuda(), adj[1].cuda())
    entries = adj[1].numel()
    man, table = manifold_and_table(sb, "upper", 2, "riem", n, seed=6)
    t = table.cuda()
    block_bytes = 64 << 20
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.memory_allocated()
    est = estimate(man, t, adj, 3000, scale=1.1, block_bytes=block_bytes)
    growth = torch.cuda.max_memory_allocated() - before
    # the kernels' workspaces (kept per device, allocated by the first call that needs them)
    workspaces = sum(w.numel() * w.element_size() for cache in (ops._hop_workspace, ops._ap_workspace, ops._idx_workspace)
                     for w in cache.values())
    # estimate's docstring: the block, the workspaces, one permuted table, the relabelled adjacency, the
    # permutation and the transient index arrays; 128 bytes per node cover the per-row outputs and small tensors
    bound = (block_bytes + workspaces + t.numel() * 8 + 8 * (n + 1 + entries) + 8 * n + 48 * n + 24 * entries
             + 128 * n)
    assert growth <= bound, (growth, bound)
    assert est.distortion.count.sum().item() == 3000 * (n - 1)                      # a tree is connected


def test_bad_arguments(sb):
    from sympa_b200.metrics import estimate
    adj, rows = product_graph(sb)
    man, table = manifold_and_table(sb, "upper", 2, "riem", rows, seed=0)
    with pytest.raises(ValueError):
        estimate(man, table.cuda(), adj, rows + 1)
    with pytest.raises(ValueError):
        estimate(man, table.cuda(), adj, 0)
    with pytest.raises(ValueError):
        estimate(man, table.cuda(), adj, 4, seed=-1)
    with pytest.raises(RuntimeError, match="no CPU path"):
        estimate(man, table, adj, 4)


def test_model_estimate_uses_its_own_scale(sb):
    from sympa_b200.metrics import estimate
    from sympa_b200.model import Model
    adj, rows = product_graph(sb)
    args = types.SimpleNamespace(manifold="upper", metric="riem", dims=3, num_points=rows, scale_init=1.6, scale_coef=1.0,
                                 train_scale=True)
    model = Model(args).cuda()
    model.embeddings.embeds.data.copy_(so.upper_spread(rows, 3, generator=torch.Generator().manual_seed(0)).cuda())
    got = model.estimate(adj, 40, seed=2)
    want = estimate(model.manifold, model.embeddings.embeds, adj, 40, scale=float(model.get_scale()), seed=2)
    assert got[:5] == want[:5] and same(got.ap, want.ap) and same_rows(got.distortion, want.distortion)
    full = model.estimate(adj, rows)
    avg, m_ap = model.evaluate(adj)
    assert full.average_distortion == pytest.approx(avg, rel=1e-12) and full.mean_ap == pytest.approx(m_ap, rel=1e-12)
