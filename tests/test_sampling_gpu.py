"""The pair sampler on the device (sympa_sample_pairs, ops.sample_pairs, sampling.PairSampler): bit for bit equal to
the Python oracle on the graphs of test_distortion_gpu.py, the config-3 product graph and a 2^20-node random tree
(the visited set in global memory), for K below and above the reachable count; invariant to how the sources are
split, ordered, repeated or sharded over ranks; both status bits; a workspace independent of the source count; and
training on sampled pairs through the existing trainers."""
import ctypes
import functools
import types

import numpy as np
import pytest
import torch

import sampling_oracle as oracle
from distortion_oracle import hop_matrix
from test_distortion_gpu import graph_case, random_tree

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb():
    if not torch.cuda.is_available():
        pytest.skip("needs CUDA")
    import sympa_b200
    import sympa_b200.graphs  # noqa: F401
    import sympa_b200.sampling  # noqa: F401
    from sympa_b200 import _lib
    _lib.load()
    return sympa_b200


GRAPHS = ["components", "path", "star", "grid", "config3", "random_tree_2_20"]


@functools.lru_cache(maxsize=None)
def graph_with_sources(name):
    """(ptr, idx) on the CPU, N, the sources to sample from and their hop rows (scipy)"""
    import sympa_b200.graphs as graphs
    rng = np.random.default_rng(21)
    if name == "config3":
        ids, gd, n = graphs.product_cartesian_triplets(3, 3, 5, 3)
        adj = graphs.adjacency_csr(ids[gd == 1], n)
    elif name == "random_tree_2_20":
        n = 1 << 20
        adj = graphs.adjacency_csr(torch.from_numpy(random_tree(rng, n)), n)
    else:
        adj, n = graph_case(types.SimpleNamespace(graphs=graphs), name)
    count = 6 if name == "random_tree_2_20" else 40
    sources = rng.choice(n, count, replace=False)
    if name == "components":
        sources[:3] = (545, 0, 556)           # two isolated nodes (no pair) among them
    if name == "star":
        sources[0] = 0                         # the hub
    uniq, inv = np.unique(sources, return_inverse=True)
    rows = hop_matrix(adj[0].numpy(), adj[1].numpy(), rows=uniq)[inv]
    return adj, n, sources.astype(np.int64), rows


def clear_status(sb):
    sb.ops.status_word(torch.device("cuda", torch.cuda.current_device())).zero_()


def on_device(adj):
    return adj[0].cuda(), adj[1].cuda()


@pytest.mark.parametrize("k", [1, 7, 1000])
@pytest.mark.parametrize("name", GRAPHS)
def test_sample_pairs_equal_the_oracle_bit_for_bit(sb, name, k):
    adj, n, sources, rows = graph_with_sources(name)
    seed, epoch = 0x5EED + k, 3
    want_ids, want_d = oracle.pairs_from_rows(rows, sources, k, seed, epoch)
    clear_status(sb)
    ids, d = sb.ops.sample_pairs(on_device(adj), torch.from_numpy(sources).cuda(), k, seed, epoch)
    if name == "components":
        with pytest.raises(AssertionError, match="reaches no other node"):
            sb.ops.check_status()
    sb.ops.check_status()
    assert ids.shape == (len(sources) * k, 2) and ids.dtype == torch.int64 and d.dtype == torch.float64
    np.testing.assert_array_equal(ids.cpu().numpy(), want_ids)
    assert np.array_equal(d.cpu().numpy().view(np.int64), want_d.view(np.int64))
    if k == 1000:
        # K above the reachable count of some sources: draws repeat, every reachable node of a small component occurs
        reach = (rows >= 1).sum(1)
        small = np.flatnonzero((reach > 0) & (reach < 50))
        for i in small:
            got = set(want_ids[i * k:(i + 1) * k, 1].tolist())
            assert got == set(np.flatnonzero(rows[i] >= 1).tolist())


def test_other_seeds_and_epochs_draw_other_pairs(sb):
    adj, n, sources, rows = graph_with_sources("grid")
    src = torch.from_numpy(sources).cuda()
    a = sb.ops.sample_pairs(on_device(adj), src, 64, 1, 0)[0]
    for seed, epoch in ((2, 0), (1, 1), ((1 << 64) - 1, (1 << 64) - 1)):
        b = sb.ops.sample_pairs(on_device(adj), src, 64, seed, epoch)[0]
        assert torch.equal(a[:, 0], b[:, 0]) and not torch.equal(a[:, 1], b[:, 1])
        want, _ = oracle.pairs_from_rows(rows, sources, 64, seed, epoch)
        np.testing.assert_array_equal(b.cpu().numpy(), want)
    sb.ops.check_status()


@pytest.mark.parametrize("name", ["components", "random_tree_2_20"])
def test_split_reordered_and_repeated_source_lists(sb, name):
    adj, n, sources, _ = graph_with_sources(name)
    dev_adj = on_device(adj)
    k = 9

    def run(src):
        return sb.ops.sample_pairs(dev_adj, torch.as_tensor(src, dtype=torch.int64).cuda(), k, 4, 2)

    ids, d = run(sources)
    blocks = ids.reshape(len(sources), k, 2), d.reshape(len(sources), k)
    cut = len(sources) // 3
    a, b = run(sources[:cut]), run(sources[cut:])
    assert torch.equal(torch.cat((a[0], b[0])), ids) and torch.equal(torch.cat((a[1], b[1])), d)
    perm = np.random.default_rng(1).permutation(len(sources))
    p = run(sources[perm])
    assert torch.equal(p[0].reshape(-1, k, 2), blocks[0][torch.from_numpy(perm).cuda()])
    assert torch.equal(p[1].reshape(-1, k), blocks[1][torch.from_numpy(perm).cuda()])
    rep = np.repeat(sources[:4], 3)
    r = run(rep)
    assert torch.equal(r[0].reshape(-1, k, 2), blocks[0][:4].repeat_interleave(3, 0))
    if name == "components":                    # its isolated sources
        with pytest.raises(AssertionError, match="reaches no other node"):
            sb.ops.check_status()
    sb.ops.check_status()


@pytest.mark.parametrize("world", [2, 3])
def test_rank_shards_union_to_one_call(sb, world):
    from sympa_b200.sampling import PairSampler
    adj, n, _, _ = graph_with_sources("config3")
    sampler = PairSampler(on_device(adj), 301, 17, seed=8)
    full_src = sampler.epoch_sources(5)
    ids, d = sampler.sample(5)
    assert torch.equal(ids, sb.ops.sample_pairs(sampler.adj, full_src, 17, 8, 5)[0])
    by_source = {}
    for rank in range(world):
        src = sampler.epoch_sources(5, rank, world)
        r_ids, r_d = sampler.sample(5, rank, world)
        assert r_ids.shape[0] == sampler.pairs_per_rank(world) == -(-301 // world) * 17
        for i, u in enumerate(src.tolist()):
            by_source.setdefault(u, []).append((r_ids[i * 17:(i + 1) * 17], r_d[i * 17:(i + 1) * 17]))
    assert sorted(by_source) == sorted(full_src.tolist())
    for i, u in enumerate(full_src.tolist()):
        for r_ids, r_d in by_source[u]:          # a padded source appears twice, with the same pairs
            assert torch.equal(r_ids, ids[i * 17:(i + 1) * 17]) and torch.equal(r_d, d[i * 17:(i + 1) * 17])
    sb.ops.check_status()


def test_out_of_range_source_sets_bad_index(sb):
    adj, n, _, _ = graph_with_sources("path")
    src = torch.tensor([5, -1, n, 7], dtype=torch.int64).cuda()
    clear_status(sb)
    ids, d = sb.ops.sample_pairs(on_device(adj), src, 4, 0, 0)
    with pytest.raises(AssertionError, match="out of range") as e:
        sb.ops.check_status()
    assert "reaches no other node" not in str(e.value)
    assert ids[4:12].tolist() == [[-1, -1]] * 4 + [[n, n]] * 4 and d[4:12].tolist() == [0.0] * 8
    good, _ = sb.ops.sample_pairs(on_device(adj), src[[0, 3]], 4, 0, 0)
    assert torch.equal(ids[:4], good[:4]) and torch.equal(ids[12:], good[4:])
    sb.ops.check_status()


def test_isolated_source_sets_no_pair(sb):
    import sympa_b200.graphs as graphs
    adj = on_device(graphs.adjacency_csr(torch.tensor([[0, 1], [2, 2]]), 4))    # 2 has only a self loop (removed)
    clear_status(sb)
    ids, d = sb.ops.sample_pairs(adj, torch.tensor([3, 1, 2]).cuda(), 2, 0, 0)
    with pytest.raises(AssertionError, match="reaches no other node"):
        sb.ops.check_status()
    assert ids.tolist() == [[3, 3], [3, 3], [1, 0], [1, 0], [2, 2], [2, 2]] and d.tolist() == [0, 0, 1, 1, 0, 0]


def test_workspace_does_not_grow_with_the_source_count(sb):
    from sympa_b200 import _lib, ops
    lib = _lib.load()
    adj, n, _, _ = graph_with_sources("random_tree_2_20")
    dev_adj = on_device(adj)
    nbytes = lib.sympa_sample_pairs_workspace_bytes(n)
    assert nbytes == lib.sympa_sample_pairs_workspace_bytes(n)
    assert nbytes < 12 * n * torch.cuda.get_device_properties(0).multi_processor_count * 2 + 4096
    ops.sample_pairs(dev_adj, torch.tensor([0]).cuda(), 1, 0, 0)
    ws = ops._sample_workspace[(("cuda", torch.cuda.current_device()))]
    assert ws.numel() * 8 >= nbytes
    src = torch.randint(0, n, (4096,)).cuda()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.memory_allocated()
    ids, d = ops.sample_pairs(dev_adj, src, 3, 0, 0)
    growth = torch.cuda.max_memory_allocated() - before
    assert ops._sample_workspace[("cuda", torch.cuda.current_device())] is ws
    assert growth <= ids.numel() * 8 + d.numel() * 8 + (1 << 20), growth
    ops.check_status()


def test_bad_arguments(sb):
    from sympa_b200 import _lib
    lib = _lib.load()
    import sympa_b200.graphs as graphs
    ptr, idx = on_device(graphs.adjacency_csr(torch.tensor([[0, 1], [1, 2]]), 3))
    src = torch.tensor([0, 2]).cuda()
    with pytest.raises(RuntimeError, match="no CPU path"):
        sb.ops.sample_pairs((ptr.cpu(), idx.cpu()), src.cpu(), 2, 0, 0)
    with pytest.raises(TypeError):
        sb.ops.sample_pairs((ptr, idx), src.int(), 2, 0, 0)
    with pytest.raises(ValueError):
        sb.ops.sample_pairs((ptr, idx), src, -1, 0, 0)
    with pytest.raises(ValueError):
        sb.ops.sample_pairs((ptr, idx), src, 2, -1, 0)
    with pytest.raises(ValueError):
        sb.ops.sample_pairs((ptr, idx), src, 2, 0, 1 << 64)
    with pytest.raises(ValueError):
        sb.ops.sample_pairs((ptr, idx), src.reshape(2, 1), 2, 0, 0)
    with pytest.raises(ValueError):
        sb.ops.sample_pairs((ptr, idx), src, 2, 0, 0, out=(torch.empty(4, 2, dtype=torch.int64, device="cuda"),
                                                            torch.empty(3, dtype=torch.float64, device="cuda")))
    empty = sb.ops.sample_pairs((ptr, idx), src[:0], 5, 0, 0)
    assert empty[0].shape == (0, 2) and empty[1].shape == (0,)
    P = ctypes.c_void_p
    nbytes = lib.sympa_sample_pairs_workspace_bytes(3)
    assert nbytes > 256 and lib.sympa_sample_pairs_workspace_bytes(-1) == -1
    assert lib.sympa_sample_pairs_workspace_bytes(1 << 31) == -1
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    ids = torch.empty(4, 2, dtype=torch.int64, device="cuda")
    d = torch.empty(4, dtype=torch.float64, device="cuda")
    a = (P(ptr.data_ptr()), P(idx.data_ptr()))
    o = (P(ids.data_ptr()), P(d.data_ptr()), P(ws.data_ptr()))
    assert lib.sympa_sample_pairs(3, *a, 2, P(src.data_ptr()), 2, 1, 2, *o, nbytes, None, None) == 0
    assert lib.sympa_sample_pairs(3, *a, 2, P(src.data_ptr()), -2, 1, 2, *o, nbytes, None, None) == 1
    assert lib.sympa_sample_pairs(3, *a, -2, P(src.data_ptr()), 2, 1, 2, *o, nbytes, None, None) == 1
    assert lib.sympa_sample_pairs(3, *a, 2, P(src.data_ptr()), 2, 1, 2, *o, nbytes - 1, None, None) == 1
    assert lib.sympa_sample_pairs(3, *a, 2, None, 2, 1, 2, *o, nbytes, None, None) == 1
    assert lib.sympa_sample_pairs(3, *a, 2, P(src.data_ptr()), 1 << 62, 1, 2, *o, nbytes, None, None) == 1
    torch.cuda.synchronize()
    want, want_d = oracle.sample_pairs(ptr.cpu().numpy(), idx.cpu().numpy(), [0, 2], 2, 1, 2)
    assert ids.cpu().tolist() == want.tolist() and d.cpu().tolist() == want_d.tolist()


# ------------------------------------------------------------------------------------------- training
def tree_model(sb, manifold="bounded", metric="fone", dims=3, seed=0):
    from sympa_b200.model import Model
    args = types.SimpleNamespace(manifold=manifold, metric=metric, dims=dims, num_points=364, scale_init=1.0,
                                 scale_coef=1.0, train_scale=False)
    torch.manual_seed(seed)
    return Model(args).cuda()


def tree_adj(sb):
    import sympa_b200.graphs as graphs
    k = torch.arange(1, 364)
    return on_device(graphs.adjacency_csr(torch.stack((k, (k - 1) // 3), 1), 364))


def close_tables(a, b):
    # the table-gradient scatter adds with FP64 atomics, whose order between two runs is not fixed: equal pairs give
    # equal tables up to that rounding
    torch.testing.assert_close(a, b, rtol=1e-10, atol=1e-13)


def test_fused_runner_fed_in_place_equals_fresh_runners(sb):
    from sympa_b200.runner import FusedEpochRunner
    from sympa_b200.sampling import PairSampler
    sampler = PairSampler(tree_adj(sb), 200, 24, seed=3)
    fed = tree_model(sb)
    fresh = tree_model(sb)
    assert torch.equal(fed.embeddings.embeds, fresh.embeddings.embeds)
    ids, gd = sampler.sample(0)
    runner = FusedEpochRunner(fed, 5e-2, ids, gd, 512, max_grad_norm=3.0)
    for epoch in range(3):
        got = sampler.sample(epoch, out=(runner.ids, runner.gdist))
        assert got[0] is runner.ids and got[1] is runner.gdist
        runner.run_epoch(epoch)
        e_ids, e_gd = (t.clone() for t in sampler.sample(epoch))
        other = FusedEpochRunner(fresh, 5e-2, e_ids, e_gd, 512, max_grad_norm=3.0)
        other.run_epoch(epoch)
        # the epoch's pairs reached both runners' buffers bit for bit
        assert torch.equal(runner.idx_buf, other.idx_buf) and torch.equal(runner.gd_buf, other.gd_buf)
        close_tables(fed.embeddings.embeds.detach(), fresh.embeddings.embeds.detach())
    assert not torch.equal(fed.embeddings.embeds, tree_model(sb).embeddings.embeds)


def test_presharded_on_one_rank_is_the_default(sb):
    from sympa_b200.optim import RiemannianSGD
    from sympa_b200.runner import FusedEpochRunner, train_epoch
    from sympa_b200.sampling import PairSampler
    sampler = PairSampler(tree_adj(sb), 150, 16, seed=5)
    ids, gd = sampler.sample(1)
    models = [tree_model(sb) for _ in range(2)]
    runners = [FusedEpochRunner(m, 5e-2, ids, gd, 256, max_grad_norm=3.0, presharded=p) for m, p in zip(models, (False, True))]
    losses = [r.run_epoch(1) for r in runners]
    assert torch.equal(runners[0].idx_buf, runners[1].idx_buf)
    assert losses[0] == pytest.approx(losses[1], rel=1e-12)
    close_tables(models[0].embeddings.embeds.detach(), models[1].embeddings.embeds.detach())
    models = [tree_model(sb) for _ in range(2)]
    losses = []
    for m, p in zip(models, (False, True)):
        opt = RiemannianSGD(m.parameters(), lr=5e-2, fused=True)
        losses.append(train_epoch(m, opt, ids, gd, 256, max_grad_norm=3.0, epoch=1, presharded=p))
    assert losses[0] == pytest.approx(losses[1], rel=1e-12)
    close_tables(models[0].embeddings.embeds.detach(), models[1].embeddings.embeds.detach())


def test_distortion_falls_when_training_on_sampled_pairs(sb):
    """config 2's tree (364 nodes, bounded fone n = 3), trained only from sampled pairs"""
    from sympa_b200.runner import FusedEpochRunner
    from sympa_b200.sampling import PairSampler
    adj = tree_adj(sb)
    model = tree_model(sb, seed=1)
    sampler = PairSampler(adj, 364, 32, seed=11)
    before, _ = model.evaluate(adj)
    ids, gd = sampler.sample(0)
    runner = FusedEpochRunner(model, 5e-2, ids, gd, 512, max_grad_norm=3.0)
    curve = [before]
    for epoch in range(6):
        sampler.sample(epoch, out=(runner.ids, runner.gdist))
        runner.run_epoch(epoch)
        if epoch % 2 == 1:
            curve.append(model.evaluate(adj)[0])
    # on a B200: 0.9994, 0.961, 0.906, 0.870 - falling at every check
    assert all(np.isfinite(curve)) and all(b < a for a, b in zip(curve, curve[1:])), curve
    assert curve[-1] < 0.92 * curve[0], curve
