"""Link-prediction evaluation on the device (sympa_target_ranks, sympa_b200.metrics.link_prediction): the count kernel
exactly against the numpy definition (rank_oracle) on blocks with heavy ties, signed zeros, inf, NaN rows, hub rows
and out-of-range filter entries, at every block height and offset; link_prediction against the oracle on the rows of
the distance matrix for every kind, invariant to the block size and the rank shards; agreement with the exact k-NN
path; Model.link_prediction."""
import ctypes
import math
import types

import numpy as np
import pytest
import torch

import rank_oracle
import siegel_oracle as so

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    import sympa_b200
    import sympa_b200.metrics  # noqa: F401
    from sympa_b200 import _lib
    _lib.load()
    return sympa_b200


def status_bits():
    from sympa_b200 import ops
    w = ops.status_word(torch.device("cuda", torch.cuda.current_device()))
    v = int(w.item())
    w.zero_()
    return v


def csr_from_rows(rows):
    """(ptr, idx) int64 numpy arrays of a list of per-row id lists"""
    ptr = np.zeros(len(rows) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum([len(r) for r in rows])
    idx = np.array([w for r in rows for w in r], dtype=np.int64)
    return ptr, idx


def synthetic_case(rng):
    """(block, queries, targets CSR, filter CSR) over N = 5000 columns: five distance levels with signed zeros, a
    row of +-inf, NaN rows, rows without targets, a row of 3000 targets, a query whose filter row has 3000 entries and
    filter rows with out-of-range entries (sorted in, as -3 and N + 5)"""
    n_cols, rows = 5000, 24
    block = rng.integers(0, 5, (rows, n_cols)).astype(np.float64) * 0.25 - 0.5
    zeros = block == 0.0
    block[zeros] = np.where(rng.random(zeros.sum()) < 0.5, -0.0, 0.0)
    block[2, rng.integers(0, n_cols, 50)] = np.inf
    block[2, rng.integers(0, n_cols, 50)] = -np.inf
    block[5, 17] = np.nan                                   # one NaN entry: the whole row is undefined
    block[6] = np.nan
    block[8] = rng.random(n_cols)                           # no ties
    block[9] = 1.0                                          # all equal
    queries = rng.choice(n_cols, rows, replace=False)
    block[3, queries[3]] = np.nan                           # on the diagonal: not a competitor, the row stays defined
    t_rows = []
    for r in range(rows):
        cand = np.setdiff1d(np.arange(n_cols), [queries[r]])
        m = {1: 0, 4: 0, 7: 3000, 10: 1}.get(r, int(rng.integers(1, 40)))
        t = list(rng.choice(cand, m, replace=m > cand.size))
        if r == 11:
            t += t[:3]                                      # a target listed twice
        t_rows.append(t)
    f_rows = [[] for _ in range(n_cols)]
    for r in range(rows):
        u = int(queries[r])
        size = 3000 if r == 12 else int(rng.integers(0, 60))
        f = sorted(set(rng.choice(n_cols, size, replace=False).tolist()) - {u})
        if r in (12, 13):
            f.append(u)                                     # the node itself: ignored
            f = sorted(f)
        if r in (13, 14):
            f = [-3] + f + [n_cols + 5]                     # out of range: skipped
        if r == 15 and t_rows[r]:
            f = sorted(set(f) | set(t_rows[r][:2]))         # some targets are known edges themselves
        f_rows[u] = f
    return block, queries, csr_from_rows(t_rows), csr_from_rows(f_rows)


def oracle_counts(block, queries, targets, filt):
    t_ptr, t_idx = targets
    f_ptr, f_idx = filt
    lt = np.full(t_idx.size, -1, dtype=np.int64)
    le = np.full(t_idx.size, -1, dtype=np.int64)
    for r, u in enumerate(queries.tolist()):
        f = f_idx[f_ptr[u]:f_ptr[u + 1]].tolist()
        for i in range(t_ptr[r], t_ptr[r + 1]):
            lt[i], le[i] = rank_oracle.counts(block[r], u, int(t_idx[i]), f)
    return lt, le


def test_target_ranks_equal_the_definition_at_every_block(sb):
    from sympa_b200 import ops
    rng = np.random.default_rng(0)
    block, queries, targets, filt = synthetic_case(rng)
    want = oracle_counts(block, queries, targets, filt)
    d = torch.from_numpy(block).cuda()
    q = torch.from_numpy(queries).cuda()
    t = tuple(torch.from_numpy(a).cuda() for a in targets)
    f = tuple(torch.from_numpy(a).cuda() for a in filt)
    status_bits()
    lt, le = ops.target_ranks(d, q, t, f)
    assert lt.cpu().tolist() == want[0].tolist() and le.cpu().tolist() == want[1].tolist()
    assert status_bits() == 8 | 16                         # the NaN rows and the out-of-range filter entries
    # a pair's result does not depend on the block it comes in or where that block starts
    ptr = targets[0]
    rows = d.shape[0]
    for height in (1, 3, 16):
        for r0 in range(rows):
            r1 = min(rows, r0 + height)
            out = (torch.full_like(t[1], -7), torch.full_like(t[1], -7))
            ops.target_ranks(d[r0:r1], q[r0:r1], (t[0][r0:r1 + 1], t[1]), f, out=out)
            inside = np.zeros(t[1].numel(), dtype=bool)
            inside[ptr[r0]:ptr[r1]] = True
            for got, exp in zip(out, want):
                got = got.cpu().numpy()
                assert (got[inside] == exp[inside]).all() and (got[~inside] == -7).all(), (height, r0)
    status_bits()


def test_target_ranks_without_a_filter_and_with_a_short_workspace(sb):
    from sympa_b200 import _lib, ops
    rng = np.random.default_rng(1)
    block, queries, targets, _ = synthetic_case(rng)
    n_cols = block.shape[1]
    raw = (np.zeros(n_cols + 1, dtype=np.int64), np.zeros(0, dtype=np.int64))
    want = oracle_counts(block, queries, targets, raw)
    d = torch.from_numpy(block).cuda()
    q = torch.from_numpy(queries).cuda()
    t = tuple(torch.from_numpy(a).cuda() for a in targets)
    f = tuple(torch.from_numpy(a).cuda() for a in raw)
    lt, le = ops.target_ranks(d, q, t, f)
    assert lt.cpu().tolist() == want[0].tolist() and le.cpu().tolist() == want[1].tolist()
    status_bits()
    # a workspace with room for the first rows' targets only: the others get -1 and the out-of-range bit
    lib = _lib.load()
    rows = d.shape[0]
    room = int(targets[0][6])
    ws = torch.empty(rows + 3 * room, dtype=torch.float64, device="cuda")
    lt, le = torch.full_like(t[1], -7), torch.full_like(t[1], -7)
    P = ctypes.c_void_p
    w = ops.status_word(d.device)
    assert lib.sympa_target_ranks(rows, n_cols, P(d.data_ptr()), P(q.data_ptr()), P(t[0].data_ptr()), P(t[1].data_ptr()),
                                  P(f[0].data_ptr()), P(t[1].data_ptr()), P(lt.data_ptr()), P(le.data_ptr()),
                                  P(ws.data_ptr()), ws.numel() * 8, P(w.data_ptr()), None) == 0
    assert lt[:room].cpu().tolist() == want[0][:room].tolist()
    assert (lt[room:] == -1).all() and (le[room:] == -1).all()
    assert status_bits() & 16
    assert lib.sympa_target_ranks_workspace_bytes(3, 10) == 8 * (3 + 30)
    assert lib.sympa_target_ranks_workspace_bytes(-1, 10) == -1
    assert lib.sympa_target_ranks(rows, n_cols, P(d.data_ptr()), P(q.data_ptr()), P(t[0].data_ptr()), P(t[1].data_ptr()),
                                  P(f[0].data_ptr()), P(t[1].data_ptr()), P(lt.data_ptr()), P(le.data_ptr()),
                                  P(ws.data_ptr()), 8 * rows - 8, None, None) == 1


def test_target_ranks_of_bad_targets_and_queries(sb):
    from sympa_b200 import ops
    block = np.array([[0.0, 1.0, 2.0, 2.0], [3.0, 0.0, 1.0, 1.0]])
    d = torch.from_numpy(block).cuda()
    f = (torch.zeros(5, dtype=torch.int64, device="cuda"), torch.zeros(0, dtype=torch.int64, device="cuda"))
    t = (torch.tensor([0, 3, 5], device="cuda"), torch.tensor([2, 9, -1, 3, 0], device="cuda"))
    status_bits()
    lt, le = ops.target_ranks(d, torch.tensor([0, 1], device="cuda"), t, f)
    assert lt.tolist() == [1, -1, -1, 0, 2] and le.tolist() == [2, -1, -1, 1, 2]
    assert status_bits() == 16
    lt, le = ops.target_ranks(d, torch.tensor([0, 4], device="cuda"), t, f)       # a query outside the table
    assert lt.tolist() == [1, -1, -1, -1, -1]
    assert status_bits() == 16
    with pytest.raises(ValueError, match="R \\+ 1"):
        ops.target_ranks(d, torch.tensor([0, 1], device="cuda"), (t[0][:2], t[1]), f)
    with pytest.raises(ValueError, match="N \\+ 1"):
        ops.target_ranks(d, torch.tensor([0, 1], device="cuda"), t, (f[0][:3], f[1]))


METRICS = ["riem", "finf"]
CASES = ([(kind, n, m) for kind in ("upper", "bounded") for n in (2, 4, 7, 10) for m in METRICS]
         + [("spd", n, "riem") for n in (2, 4, 7, 10)])
ROWS = 97


def manifold_and_table(sb, kind, n, metric, rows, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "spd":
        return sb.SymmetricPositiveDefinite().cuda(), so.spd_spread(rows, n, generator=g).cuda()
    table = so.upper_spread(rows, n, generator=g, scale=0.3)
    if kind == "bounded":
        table = so.to_symmetric(so.cayley_transform(table))
    cls = {"upper": sb.UpperHalfManifold, "bounded": sb.BoundedDomainManifold}[kind]
    return cls(dims=n, metric=sb.MetricType.from_str(metric)).cuda(), table.cuda()


def route_matrix(man, t):
    """the matrix link_prediction ranks on: dist_matrix of the table, or of the bounded domain's inverse Cayley
    transform (the route evaluate and nearest take)"""
    from sympa_b200 import metrics, ops
    src, kind, metric, wsum = metrics._distance_source(man, t)
    return ops.dist_matrix(kind, metric, src, wsum_w=wsum)


def held_out(sb, n_nodes, n_edges, seed, fraction=0.2):
    """(test pairs in both directions, filter = the whole graph) of a random graph"""
    from sympa_b200 import graphs
    edges = torch.from_numpy(np.random.default_rng(seed).integers(0, n_nodes, (n_edges, 2)))
    _, test = graphs.split_edges(edges, n_nodes, fraction, seed=seed)
    return torch.cat((test, test.flip(1))), graphs.adjacency_csr(edges, n_nodes)


def assert_matches_oracle(res, pairs, d, filt, ks):
    lt, le = rank_oracle.pair_counts(d, pairs.cpu().numpy(), filt[0].cpu().numpy(), filt[1].cpu().numpy())
    want = rank_oracle.ranks(lt, le)
    assert res.pairs.cpu().tolist() == list(range(pairs.shape[0]))
    for got, exp in zip((res.rank, res.optimistic, res.pessimistic), want):
        assert got.cpu().tolist() == exp.tolist()
    assert res.count == pairs.shape[0]
    assert math.isclose(res.mrr, float(np.mean(1.0 / want[0])), rel_tol=1e-13)
    for k in ks:
        assert res.hits[k] == float(np.mean(want[0] <= k))


@pytest.mark.parametrize("kind,n,metric", CASES)
def test_link_prediction_equals_the_oracle_on_the_matrix_rows(sb, kind, n, metric):
    from sympa_b200.metrics import link_prediction
    man, t = manifold_and_table(sb, kind, n, metric, ROWS, seed=n + 11)
    d = route_matrix(man, t).cpu().numpy()
    pairs, filt = held_out(sb, ROWS, 300, seed=n)
    ks = (1, 3, 10, 50)
    res = link_prediction(man, t, pairs.cuda(), filt, ks=ks)
    assert res.rank.is_cuda and res.rank.dtype == torch.float64
    assert_matches_oracle(res, pairs, d, filt, ks)
    # the raw setting: an adjacency without edges
    from sympa_b200 import graphs
    raw = graphs.adjacency_csr(torch.zeros(0, 2, dtype=torch.int64), ROWS)
    assert_matches_oracle(link_prediction(man, t, pairs, raw, ks=ks), pairs, d, raw, ks)


def test_link_prediction_does_not_depend_on_blocks_or_shards(sb, monkeypatch):
    import torch.distributed as dist
    from sympa_b200.metrics import link_prediction
    rows = 3000
    man, t = manifold_and_table(sb, "bounded", 4, "finf", rows, seed=8)
    pairs, filt = held_out(sb, rows, 12000, seed=8, fraction=0.1)
    perm = torch.randperm(pairs.shape[0], generator=torch.Generator().manual_seed(3))
    pairs = torch.cat((pairs[perm], pairs[:40])).cuda()                # shuffled, with repeated pairs
    one = link_prediction(man, t, pairs, filt)
    d = route_matrix(man, t).cpu().numpy()
    first = pairs[:200].cpu().numpy()
    lt, le = rank_oracle.pair_counts(d, first, filt[0].numpy(), filt[1].numpy())
    assert one.rank[:200].cpu().tolist() == rank_oracle.ranks(lt, le)[0].tolist()
    for block_bytes in (8 * rows, 8 * rows * 7, 8 * rows * 300):
        again = link_prediction(man, t, pairs, filt, block_bytes=block_bytes)
        assert torch.equal(again.rank, one.rank) and torch.equal(again.pairs, one.pairs)
        assert again.mrr == one.mrr and again.hits == one.hits
    monkeypatch.setattr(dist, "all_reduce", lambda tensor, op=None: None)
    parts = [link_prediction(man, t, pairs, filt, world_size=3, rank=r, block_bytes=8 * rows * 40) for r in range(3)]
    positions = torch.cat([p.pairs for p in parts])
    assert sorted(positions.tolist()) == list(range(pairs.shape[0]))
    for field in ("rank", "optimistic", "pessimistic"):
        merged = torch.empty_like(one.rank)
        merged[positions] = torch.cat([getattr(p, field) for p in parts])
        assert torch.equal(merged, getattr(one, field))
    assert sum(p.count for p in parts) == one.count
    # each rank evaluates distinct query nodes
    sources = [set(pairs[p.pairs, 0].tolist()) for p in parts]
    assert not (sources[0] & sources[1] or sources[0] & sources[2] or sources[1] & sources[2])


def test_ranks_agree_with_nearest(sb):
    """tie-free random table, no filter: a target at position p of nearest(u, k) has rank 1 + p"""
    from sympa_b200 import graphs
    from sympa_b200.metrics import link_prediction, nearest
    rows, k = 4000, 64
    man, t = manifold_and_table(sb, "upper", 3, "riem", rows, seed=5)
    rng = np.random.default_rng(5)
    queries = torch.from_numpy(rng.choice(rows, 200, replace=False)).cuda()
    nn = nearest(man, t, queries, k)
    pick = torch.from_numpy(rng.integers(0, k, queries.numel())).cuda()
    near_targets = nn.ids.gather(1, pick[:, None])[:, 0]
    far = torch.from_numpy(rng.integers(0, rows, queries.numel())).cuda()
    far = torch.where(far == queries, (far + 1) % rows, far)
    pairs = torch.cat((torch.stack((queries, near_targets), 1), torch.stack((queries, far), 1)))
    raw = graphs.adjacency_csr(torch.zeros(0, 2, dtype=torch.int64), rows)
    res = link_prediction(man, t, pairs, raw)
    assert torch.equal(res.optimistic, res.pessimistic)                   # no ties
    checked = 0
    for i, (u_pos, v) in enumerate(zip(list(range(queries.numel())) * 2, pairs[:, 1].tolist())):
        hit = (nn.ids[u_pos] == v).nonzero()
        if hit.numel():
            assert res.rank[i].item() == 1.0 + hit.item()
            checked += 1
        else:
            assert res.rank[i].item() > k
    assert checked >= queries.numel()


def test_link_prediction_of_no_pairs_and_nan_tables(sb):
    from sympa_b200 import graphs
    from sympa_b200.metrics import link_prediction
    man, t = manifold_and_table(sb, "upper", 2, "riem", 50, seed=2)
    filt = graphs.adjacency_csr(torch.tensor([[0, 1]]), 50)
    none = link_prediction(man, t, torch.zeros(0, 2, dtype=torch.int64), filt)
    assert none.count == 0 and math.isnan(none.mrr) and all(math.isnan(h) for h in none.hits.values())
    assert none.rank.shape == (0,) and none.pairs.shape == (0,)
    bad = t.clone()
    bad[7] = float("nan")
    with pytest.raises(AssertionError, match="non-finite"):
        link_prediction(man, bad, torch.tensor([[3, 4], [7, 1]]), filt)
    status_bits()


def test_model_link_prediction_is_the_function_on_its_table(sb):
    from sympa_b200.metrics import link_prediction
    from sympa_b200.model import Model
    rows = 200
    args = types.SimpleNamespace(manifold="upper", metric="riem", dims=3, num_points=rows, scale_init=1.6, scale_coef=1.0,
                                 train_scale=True)
    model = Model(args).cuda()
    model.embeddings.embeds.data.copy_(so.upper_spread(rows, 3, generator=torch.Generator().manual_seed(0)).cuda())
    pairs, filt = held_out(sb, rows, 600, seed=4)
    got = model.link_prediction(pairs, filt, ks=(1, 5))
    want = link_prediction(model.manifold, model.embeddings.embeds, pairs, filt, ks=(1, 5))
    assert torch.equal(got.rank, want.rank) and got.mrr == want.mrr and got.hits == want.hits
    assert set(got.hits) == {1, 5}
