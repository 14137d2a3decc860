"""Graph-reconstruction metrics on the device: mean average precision and distortion.

The reference evaluates by building the whole N x N distance matrix (Runner.evaluate, sympa/runner.py:124-154)
and handing it to its metric code (sympa/metrics.py), which works on every row on the host, with the graph
distances of all pairs read from the triplets preprocess.py wrote.  Here the matrix is streamed: rows are
computed in blocks (sympa_dist_matrix), and each block is reduced on the device to per-node average precision
(sympa_average_precision) and, next to the hop distances of the same rows found by breadth-first search
(sympa_hop_distances), to per-node distortion terms (sympa_distortion_rows) before the next block overwrites it.
Memory is bounded by the block, not by 8 N^2 bytes of distances plus the graph distances of every pair.

Definitions (restated - the reference's metric code is not available, so parity with it is UNPINNED), with N(u)
the graph neighbours of u, d the manifold distance, g the hop distance and s the model scale:

    AP(u) = 1/|N(u)| sum_{v in N(u)} |{v' in N(u) : d(u,v') <= d(u,v)}| / |{w != u : d(u,w) <= d(u,v)}|
    mAP   = mean of AP(u) over the nodes with |N(u)| > 0

Without ties this is what the usual argsort loop computes (sort the row, skip the node, record hits / i at the
i-th hit); with ties it is the "tied nodes rank first" value.  It does not depend on the model scale.

    g(u, w)     hop distance in the undirected graph of the CSR adjacency (graphs.adjacency_csr); pairs with
                no path are excluded from every sum
    pairs       u < w (the reference's triplets, preprocess.py:118-126), d(u, w) = row u, column w of the matrix
    delta(u, w) = |s d(u, w) - g(u, w)| / g(u, w)
    average distortion    = mean of delta over all connected pairs u < w
    worst-case distortion = max(s d / g) / min(s d / g) over the same pairs

The reference's evaluate calls model(triplets), so the distances it scores are scaled by s (Model.get_scale()).

Estimates from sampled rows (estimate), for graphs whose N^2 distances and N searches take too long to evaluate
in full.  The sample is the S nodes with the smallest (h(seed, epoch, 2, node, 0), node) - the SplitMix64 hash of
sampling.py, tag 2 (tag 1 orders the training sources, tag 0 draws their pairs) - drawn from all N nodes.  Those
nodes are relabelled 0 .. S-1 in key order (the others follow in id order) and rows [0, S) of the relabelled
table and graph go through the same pass as evaluate.  A distance comes from the same two table rows wherever
they sit and hop distances are unique, so a sampled node's AP is bit-identical to its AP in evaluate.  Each
sampled row u counts every column w != u:

    a_u = sum of delta(u, w) over the w != u connected to u,   c_u = their number   (ops.distortion_rows, full)

    mAP estimate           the mean of AP(u) over the m sampled nodes with neighbours
    its standard error     sd / sqrt(m) * sqrt(1 - m / M), sd the sample standard deviation (m - 1 in the
                           denominator) of those AP(u), M the number of nodes with neighbours (from the degrees)
    average distortion     R = sum a_u / sum c_u, the ratio estimator over the S sampled rows
    its standard error     SE^2 = (1 - S / N) sum (a_u - R c_u)^2 / ((S - 1) S cbar^2), cbar = sum c_u / S
    sampled worst case     max(s d / g) / min(s d / g) over the sampled rows' pairs: a LOWER BOUND of the
                           worst-case distortion (the extremes over a subset of the pairs), with no standard error

At S = N both standard errors are 0 and the estimates equal evaluate's values up to the order of the sums.  A
standard error that needs two units where there is one (m = 1 < M, or S = 1 < N) is NaN.

Exact k-nearest-neighbour queries (nearest): the distance rows of the query nodes (sympa_dist_rows, bit-identical
to the rows of sympa_dist_matrix) are computed in blocks and each block is reduced on the device to the k smallest
entries of every row (sympa_row_topk), in the total order (distance, node id).

Link prediction (link_prediction) - the definition is the project's own (the reference has no link-prediction code,
so parity is unpinned).  The inputs are directed query pairs (u, v), u != v, v the held-out target of u, and a filter
adjacency F (graphs.adjacency_csr; F(u) the known neighbours of u, usually the whole graph, training and held-out
edges; an adjacency without edges gives the "raw" setting).  With d row u of the distance matrix:

    C(u, v)     = {w in [0, N) : w != u, w != v, w not in F(u)}                     competitors
    lt(u, v)    = |{w in C : d(u,w) <  d(u,v)}|
    le(u, v)    = |{w in C : d(u,w) <= d(u,v)}|
    optimistic  = 1 + lt,   pessimistic = 1 + le,   rank = 1 + (lt + le) / 2          (ties split)
    MRR         = mean over the pairs of 1 / rank
    Hits@k      = mean over the pairs of [rank <= k]

-0.0 equals +0.0 and +-inf compare as usual.  A NaN anywhere in row u (w != u) makes the ranks of every pair of u
NaN, and the status check raises, as for AP.  Ranks do not depend on the model scale.  Splitting ties gives a
collapsed embedding, every distance equal, a middle rank rather than rank 1.  All counts are integers, so a pair's
ranks are exact and do not depend on the block, the rank shard or the launch shape.  Pairs are directed: to rank both
endpoints of undirected held-out edges e, pass torch.cat((e, e.flip(1))).
"""
import collections
import math

import torch

from . import distributed as sd
from . import _lib, graphs, ops, sampling

Evaluation = collections.namedtuple("Evaluation", "average_distortion worst_case_distortion mean_ap ap distortion")
Evaluation.__doc__ = """Result of evaluate(): the two distortion figures and mAP (global when world_size > 1), the (rows,)
per-node AP of this rank's rows (NaN for a node without neighbours) and their per-node ops.DistortionRows."""

Estimate = collections.namedtuple("Estimate", "mean_ap mean_ap_se average_distortion average_distortion_se "
                                              "sampled_worst_case_distortion nodes ap distortion")
Estimate.__doc__ = """Result of estimate(): the estimates of mAP and average distortion with their standard errors, and
the worst case over the sampled pairs (a lower bound of the exact one), all global when world_size > 1; `nodes` the
int64 ids of this rank's sampled nodes, `ap` their AP (NaN for a node without neighbours) and `distortion` the
ops.DistortionRows of their whole rows (every w != u), aligned with `nodes`."""

Neighbours = collections.namedtuple("Neighbours", "ids distances")
Neighbours.__doc__ = """Result of nearest(): (Q, k) int64 node ids and float64 scaled distances, row i the k nearest nodes of
queries[i] in ascending order of distance, then of id; (-1, NaN) past the selectable nodes of a row."""


def _adjacency_on(adj, device):
    ptr, idx = adj
    return (torch.as_tensor(ptr, dtype=torch.int64).to(device).contiguous(),
            torch.as_tensor(idx, dtype=torch.int64).to(device).contiguous())


def _cuda_table(who, table):
    if not isinstance(table, torch.Tensor) or not table.is_cuda:
        raise RuntimeError(f"sympa_b200: {who} needs a CUDA table (there is no CPU path)")
    return table.detach()


def _distance_source(manifold, table, perm=None):
    """(src, kind, metric, wsum) for the distance kernels, on the current device: the table (its rows in the order
    perm when given) or, for the bounded domain, its inverse Cayley transform (sympa_bounded_rows_to_upper, once per
    table) with kind "upper"; spd takes the riem kernels and no weights."""
    kind = manifold.kind
    metric = "riem" if kind == "spd" else manifold.metric.name
    wsum = None if kind == "spd" else manifold._wsum(table)
    src = table if perm is None else table.index_select(0, perm)
    if kind == "bounded":
        t = ops._require(src, "table")
        ops._check_n(t.shape[-1])
        src = torch.empty_like(t)
        _lib.check(_lib.load().sympa_bounded_rows_to_upper(t.shape[-1], t.shape[0], ops._ptr(t), ops._ptr(src),
                                                           ops._ptr(ops.status_word(t.device)), ops._stream()))
        del t
        kind = "upper"
    return src, kind, metric, wsum


def _row_pass(who, manifold, table, adj, rows, block_bytes, world_size, rank, want_ap, scale, perm=None, full=False):
    """The one streaming pass over row blocks of the distance matrix behind every metric here.  Per block:
    dist_matrix, then average_precision (want_ap) and hop_distances + distortion_rows (scale is not None) on that
    same block.  A block holds max(1, block_bytes // (bytes per entry * N)) rows, 8 bytes per entry (distances)
    plus 4 with distortion (hop distances).  perm: the table's rows are taken in this order (table[perm], before
    the bounded domain's transform, so that one table-sized copy is held); adj must then be relabelled to match.
    full: the distortion terms of whole rows (ops.distortion_rows(full=True)) instead of the columns w > u.
    Returns (sums, extremes, ap, distortion): sums = [sum_ap, count_ap] and / or [sum_delta, pairs] and extremes
    = (max, min) of s d / g, global when world_size > 1 (one SUM all-reduce, one MAX and one MIN), the per-node
    AP and DistortionRows of this rank's rows."""
    table = _cuda_table(who, table)
    dev = table.device
    n_nodes = table.shape[0]
    begin, end = (0, n_nodes) if rows is None else (int(rows[0]), int(rows[1]))
    if not 0 <= begin <= end <= n_nodes:
        raise ValueError(f"rows must be a range inside [0, {n_nodes}]")
    if world_size > 1:
        lo, hi, _ = sd.row_shard(end - begin, rank, world_size)
        begin, end = begin + lo, begin + hi
    adj = _adjacency_on(adj, dev)
    want_distortion = scale is not None
    if want_distortion:
        scale = float(scale)
    with torch.cuda.device(dev):
        src, kind, metric, wsum = _distance_source(manifold, table, perm)
        count_rows = end - begin
        entry_bytes = 12 if want_distortion else 8
        block = max(1, min(block_bytes // (entry_bytes * max(n_nodes, 1)), max(count_rows, 1)))
        buf = torch.empty(block * n_nodes, dtype=torch.float64, device=dev)
        ap = torch.empty(count_rows, dtype=torch.float64, device=dev) if want_ap else None
        dr = None
        if want_distortion:
            hop_buf = torch.empty(block * n_nodes, dtype=torch.int32, device=dev)
            dr = ops.DistortionRows(*(torch.empty(count_rows, dtype=t, device=dev)
                                      for t in (torch.float64, torch.int64, torch.float64, torch.float64)))
        for r0 in range(begin, end, block):
            rc = min(block, end - r0)
            part = slice(r0 - begin, r0 - begin + rc)
            d = buf[: rc * n_nodes].view(rc, n_nodes)
            ops.dist_matrix(kind, metric, src, r0, rc, wsum, out=d)
            if want_ap:
                ops.average_precision(d, r0, adj, out=ap[part])
            if want_distortion:
                h = ops.hop_distances(adj, r0, rc, out=hop_buf[: rc * n_nodes].view(rc, n_nodes))
                ops.distortion_rows(d, h, r0, scale, out=ops.DistortionRows(*(o[part] for o in dr)), full=full)
        sums = []
        if want_ap:
            valid = ~torch.isnan(ap)
            sums += [ap[valid].sum(), valid.sum().to(torch.float64)]
        extremes = None
        if want_distortion:
            sums += [dr.sum.sum(), dr.count.sum().to(torch.float64)]
            extremes = (torch.cat((dr.max, dr.max.new_full((1,), -math.inf))).max().reshape(1),
                        torch.cat((dr.min, dr.min.new_full((1,), math.inf))).min().reshape(1))
        sums = torch.stack(sums)
        if world_size > 1:
            import torch.distributed as dist
            dist.all_reduce(sums)
            if want_distortion:
                dist.all_reduce(extremes[0], op=dist.ReduceOp.MAX)
                dist.all_reduce(extremes[1], op=dist.ReduceOp.MIN)
        ops.check_status(dev)
        sums = sums.tolist()
        if want_distortion:
            extremes = (extremes[0].item(), extremes[1].item())
    return sums, extremes, ap, dr


def mean_average_precision(manifold, table, adj, *, rows=None, block_bytes=1 << 30, world_size=1, rank=0):
    """Per-node average precision of rows [begin, end) (`rows`, default all N) of the distance matrix of `table`
    under `manifold`, in blocks of max(1, block_bytes // (8 N)) rows; the block buffers are reused.

    adj = (ptr, idx): the CSR adjacency of all N nodes (graphs.adjacency_csr), moved to the table's device.
    The bounded domain is evaluated on its inverse Cayley transform (sympa_bounded_rows_to_upper, once per
    table) with the upper-half kernels - the route ops.table_dist takes for dense batches.
    world_size > 1: this rank evaluates its distributed.row_shard part of [begin, end), and one all-reduce of
    (sum_ap, count) over the default process group makes those two global.

    Returns (sum_ap, count, ap): the sum of AP over the nodes of the range with neighbours, their number (global
    when world_size > 1; mAP = sum_ap / count) and the (rows,) float64 per-node AP of this rank's rows, NaN
    where a node has no neighbour.  The status word is checked once, at the end."""
    (sum_ap, count), _, ap, _ = _row_pass("mean_average_precision", manifold, table, adj, rows, block_bytes, world_size,
                                          rank, True, None)
    return sum_ap, int(count), ap


def average_distortion(manifold, table, adj, *, scale=1.0, rows=None, block_bytes=1 << 30, world_size=1, rank=0):
    """Distortion terms of rows [begin, end) (`rows`, default all N) of the distance matrix of `table` under
    `manifold`, distances multiplied by `scale` (the model scale), against the hop distances of the graph
    adj = (ptr, idx) (graphs.adjacency_csr, moved to the table's device).  Rows, blocks (max(1, block_bytes //
    (12 N)) rows: distances and hop distances), the bounded domain and world_size / rank as in
    mean_average_precision; with world_size > 1 one all-reduce of (sum, count) and one each of MAX and MIN make
    the four totals global.

    Returns (sum, count, max_ratio, min_ratio, per_row): the sum of |s d - g| / g over the connected pairs u < w
    with u in the range, their number (average distortion = sum / count), the extremes of s d / g over them
    (worst-case distortion = max_ratio / min_ratio) and the ops.DistortionRows of this rank's rows.  The status
    word is checked once, at the end."""
    (total, count), (hi, lo), _, dr = _row_pass("average_distortion", manifold, table, adj, rows, block_bytes,
                                                world_size, rank, False, scale)
    return total, int(count), hi, lo, dr


def evaluate(manifold, table, adj, *, scale=1.0, rows=None, block_bytes=1 << 30, world_size=1, rank=0):
    """Both metrics of the reference's evaluation in ONE pass over the row blocks: every block of distances
    (max(1, block_bytes // (12 N)) rows) is computed once and read by the AP and the distortion kernels, so the
    distance computation is paid once.  Keywords as in average_distortion; the per-node values are bit-identical
    to those of mean_average_precision and average_distortion.  Returns an Evaluation."""
    (sum_ap, count_ap, total, pairs), (hi, lo), ap, dr = _row_pass("evaluate", manifold, table, adj, rows, block_bytes,
                                                                   world_size, rank, True, scale)
    return Evaluation(average_distortion=total / pairs if pairs else math.nan,
                      worst_case_distortion=worst_case(hi, lo) if pairs else math.nan,
                      mean_ap=sum_ap / max(count_ap, 1), ap=ap, distortion=dr)


def nearest(manifold, table, queries, k, *, scale=1.0, exclude_self=True, block_bytes=1 << 30, world_size=1, rank=0):
    """The k nearest nodes of every node in `queries` under `manifold`, exactly: a Neighbours of (Q, k) ids (int64)
    and distances (float64, multiplied by `scale`) on the table's device, nearest first.  Row i is the stable
    ascending sort of row queries[i] of the distance matrix (ties by node id, -0.0 equal to +0.0), without the query
    node itself when exclude_self, cut to k; NaN distances are never selected (the status check raises) and a row
    with fewer than k selectable nodes is padded with (-1, NaN).

    queries: 1-D int64 tensor of node ids in [0, N), repeats allowed, possibly empty; 1 <= k <= min(1024, N - 1)
    with exclude_self (N without).  Both are checked before any launch.  The queries go through in blocks of
    max(1, block_bytes // (8 N)) rows, one reused block buffer: their distance rows (ops.dist_rows, bit-identical to
    the rows of dist_matrix; the bounded domain on its inverse Cayley transform, once per table, as in evaluate),
    then the k smallest of each row (ops.row_topk).  Beyond the block it holds the (Q, k) outputs and the two
    kernels' workspaces.  world_size > 1: this rank answers its distributed.row_shard part of the queries (no
    collective).  The status word is checked once, at the end."""
    if not isinstance(table, torch.Tensor):
        raise TypeError("table must be a tensor")
    if not isinstance(queries, torch.Tensor) or queries.dtype != torch.int64:
        raise TypeError("queries must be an int64 tensor")
    if queries.dim() != 1:
        raise ValueError("queries must be 1-D")
    n_nodes = table.shape[0]
    k = int(k)
    top = min(ops.TOPK_MAX_K, n_nodes - bool(exclude_self))
    if not 1 <= k <= top:
        raise ValueError(f"k must lie in [1, {top}]" if top >= 1 else f"a table of {n_nodes} nodes has no neighbour to return")
    if queries.numel() and (int(queries.min()) < 0 or int(queries.max()) >= n_nodes):
        raise ValueError(f"queries must lie in [0, {n_nodes})")
    table = _cuda_table("nearest", table)
    dev = table.device
    if world_size > 1:
        lo, hi, _ = sd.row_shard(queries.numel(), rank, world_size)
        queries = queries[lo:hi]
    with torch.cuda.device(dev):
        queries = queries.to(dev).contiguous()
        count = queries.numel()
        ids = torch.empty(count, k, dtype=torch.int64, device=dev)
        dist = torch.empty(count, k, dtype=torch.float64, device=dev)
        if count:
            src, kind, metric, wsum = _distance_source(manifold, table)
            block = max(1, min(block_bytes // (8 * n_nodes), count))
            buf = torch.empty(block * n_nodes, dtype=torch.float64, device=dev)
            for q0 in range(0, count, block):
                qc = min(block, count - q0)
                q = queries[q0:q0 + qc]
                d = ops.dist_rows(kind, metric, src, q, wsum, out=buf[: qc * n_nodes].view(qc, n_nodes))
                ops.row_topk(d, k, exclude=q if exclude_self else None, out=(ids[q0:q0 + qc], dist[q0:q0 + qc]))
            del buf, src
            dist.mul_(float(scale))
        ops.check_status(dev)
    return Neighbours(ids, dist)


LinkPrediction = collections.namedtuple("LinkPrediction", "mrr hits count pairs rank optimistic pessimistic")
LinkPrediction.__doc__ = """Result of link_prediction(): MRR, `hits` = {k: Hits@k} and the number of pairs, global when
world_size > 1; `pairs` the int64 positions in the input of this rank's pairs, ascending, and `rank`, `optimistic`,
`pessimistic` their float64 ranks (module docstring), aligned with `pairs`."""


def link_prediction(manifold, table, pairs, filter_adj, *, ks=(1, 3, 10), block_bytes=1 << 30, world_size=1, rank=0):
    """Filtered link-prediction ranks of the directed query pairs `pairs` ((E, 2) int64 (u, v), v the held-out target
    of u, ids in [0, N), u != v) among all N nodes under `manifold`, with MRR and Hits@k for every k in `ks`, as
    defined in the module docstring.  filter_adj = (ptr, idx): the CSR adjacency (graphs.adjacency_csr) of the known
    edges left out of the competitors, moved to the table's device.  pairs, ks and the filter's N + 1 row pointers are
    checked before any launch.

    The pairs are grouped by query node on the device; the distinct query nodes go through in blocks of
    max(1, block_bytes // (8 N)) rows, one reused block buffer: their distance rows (ops.dist_rows; the bounded domain
    on its inverse Cayley transform, once per table, as in evaluate), then the counts of every target of the block's
    rows (ops.target_ranks).  Beyond the block it holds the kernels' workspaces and a few int64 / float64 arrays of E
    entries.  world_size > 1: this rank takes its distributed.row_shard part of the distinct query nodes, so no
    distance row is computed twice, and one SUM all-reduce of (sum of 1 / rank, hits per k, count) over the default
    process group makes MRR, Hits@k and count global.  The status word is checked once, at the end.  Returns a
    LinkPrediction."""
    if not isinstance(table, torch.Tensor):
        raise TypeError("table must be a tensor")
    if not isinstance(pairs, torch.Tensor) or pairs.dtype != torch.int64:
        raise TypeError("pairs must be an int64 tensor")
    if pairs.dim() != 2 or pairs.shape[1] != 2:
        raise ValueError("pairs must have shape (E, 2)")
    n_nodes = table.shape[0]
    if pairs.numel() and (int(pairs.min()) < 0 or int(pairs.max()) >= n_nodes):
        raise ValueError(f"pairs must lie in [0, {n_nodes})")
    if bool((pairs[:, 0] == pairs[:, 1]).any()):
        raise ValueError("pairs must not hold u == v")
    ks = tuple(int(k) for k in ks)
    if any(k < 1 for k in ks):
        raise ValueError("every k of ks must be >= 1")
    f_ptr, f_idx = filter_adj
    if torch.as_tensor(f_ptr).numel() != n_nodes + 1:
        raise ValueError(f"filter_adj must hold the CSR adjacency of all {n_nodes} nodes (N + 1 row pointers)")
    table = _cuda_table("link_prediction", table)
    dev = table.device
    with torch.cuda.device(dev):
        filt = _adjacency_on(filter_adj, dev)
        pairs = pairs.to(dev)
        e_all = pairs.shape[0]
        # group by query node: positions sorted by source (stable), the distinct sources with a target CSR
        order = torch.sort(pairs[:, 0], stable=True).indices
        nodes, counts = torch.unique_consecutive(pairs[order, 0], return_counts=True)
        t_ptr = torch.zeros(nodes.numel() + 1, dtype=torch.int64, device=dev)
        torch.cumsum(counts, 0, out=t_ptr[1:])
        t_idx = pairs[order, 1].contiguous()
        lo, hi = 0, nodes.numel()
        if world_size > 1:
            lo, hi, _ = sd.row_shard(nodes.numel(), rank, world_size)
        e0, e1 = (int(x) for x in t_ptr[[lo, hi]].tolist())
        lt = torch.full((e_all,), -1, dtype=torch.int64, device=dev)
        le = torch.full((e_all,), -1, dtype=torch.int64, device=dev)
        if hi > lo:
            src, kind, metric, wsum = _distance_source(manifold, table)
            block = max(1, min(block_bytes // (8 * n_nodes), hi - lo))
            buf = torch.empty(block * n_nodes, dtype=torch.float64, device=dev)
            for q0 in range(lo, hi, block):
                qc = min(block, hi - q0)
                q = nodes[q0:q0 + qc]
                d = ops.dist_rows(kind, metric, src, q, wsum, out=buf[: qc * n_nodes].view(qc, n_nodes))
                ops.target_ranks(d, q, (t_ptr[q0:q0 + qc + 1], t_idx), filt, out=(lt, le))
            del buf, src
        positions, back = torch.sort(order[e0:e1])
        lt, le = lt[e0:e1][back].to(torch.float64), le[e0:e1][back].to(torch.float64)
        undefined = lt < 0
        optimistic = (1.0 + lt).masked_fill_(undefined, math.nan)
        pessimistic = (1.0 + le).masked_fill_(undefined, math.nan)
        ranks = 1.0 + 0.5 * (lt + le)
        ranks.masked_fill_(undefined, math.nan)
        sums = torch.stack([(1.0 / ranks).sum()] + [(ranks <= k).sum().to(torch.float64) for k in ks]
                           + [torch.tensor(float(e1 - e0), dtype=torch.float64, device=dev)])
        if world_size > 1:
            import torch.distributed as dist
            dist.all_reduce(sums)
        ops.check_status(dev)
        sums = sums.tolist()
    count = int(sums[-1])
    mean = (lambda x: x / count) if count else (lambda x: math.nan)
    return LinkPrediction(mrr=mean(sums[0]), hits={k: mean(h) for k, h in zip(ks, sums[1:-1])}, count=count,
                          pairs=positions, rank=ranks, optimistic=optimistic, pessimistic=pessimistic)


def sample_order(num_nodes, num_rows, *, seed=0, epoch=0, device=None):
    """The permutation of [0, num_nodes) that estimate evaluates under: the num_rows sampled nodes first, in order of
    (h(seed, epoch, 2, node, 0), node), then the other nodes in id order.  int64 tensor on `device`."""
    nodes = torch.arange(num_nodes, dtype=torch.int64, device=device)
    keys = sampling.source_keys(seed, epoch, nodes, tag=2)
    sample = torch.sort(keys, stable=True).indices[:num_rows]         # ties: by node
    rest = torch.ones(num_nodes, dtype=torch.bool, device=device)
    rest[sample] = False
    return torch.cat((sample, nodes[rest]))


def estimate(manifold, table, adj, num_rows, *, scale=1.0, seed=0, epoch=0, block_bytes=1 << 30, world_size=1, rank=0):
    """mAP and average distortion estimated from num_rows = S sampled rows of the distance matrix of `table` under
    `manifold` (distances multiplied by `scale`), with their standard errors, as defined in the module docstring:
    S N distances and S breadth-first searches instead of N^2 and N.  The sample is sample_order(N, S, seed=seed,
    epoch=epoch); adj = (ptr, idx) as in evaluate.

    The table's rows are gathered in that order (before the bounded domain's transform) and the adjacency is
    relabelled on the device (graphs.relabel_csr); rows [0, S) then go through evaluate's pass, in blocks of
    max(1, block_bytes // (12 N)) rows, with the distortion terms of whole rows.  Beyond what evaluate holds (the
    block, the kernels' workspaces and, for the bounded domain, one transformed table), it holds one permuted
    table for the other kinds, the relabelled adjacency (8 (N + 1 + E) bytes for E adjacency entries) and, while
    sampling and relabelling, index arrays of at most 48 N + 24 E bytes.
    world_size > 1: this rank evaluates its distributed.row_shard part of the S rows; the sums the estimates need
    are all-reduced over the default process group (one SUM, MAX and MIN, then one SUM of squared deviations), so
    every figure is global.  Returns an Estimate."""
    if not isinstance(table, torch.Tensor) or not table.is_cuda:
        raise RuntimeError("sympa_b200: estimate needs a CUDA table (there is no CPU path)")
    n_nodes = table.shape[0]
    num_rows = int(num_rows)
    if not 1 <= num_rows <= n_nodes:
        raise ValueError(f"num_rows must lie in [1, {n_nodes}]")
    seed, epoch = int(seed), int(epoch)
    if not (0 <= seed < 1 << 64 and 0 <= epoch < 1 << 64):
        raise ValueError("seed and epoch must lie in [0, 2^64)")
    dev = table.device
    scale = float(scale)
    ptr, idx = _adjacency_on(adj, dev)
    if ptr.numel() != n_nodes + 1:
        raise ValueError(f"adj must hold the CSR adjacency of all {n_nodes} nodes")
    with torch.cuda.device(dev):
        perm = sample_order(n_nodes, num_rows, seed=seed, epoch=epoch, device=dev)
        relabelled = graphs.relabel_csr((ptr, idx), perm)
        with_neighbours = int((ptr[1:] > ptr[:-1]).sum())
        del ptr, idx
        (sum_ap, m, sum_a, sum_c), (hi, lo), ap, dr = _row_pass("estimate", manifold, table, relabelled, (0, num_rows),
                                                                block_bytes, world_size, rank, True, scale, perm=perm,
                                                                full=True)
        del relabelled
        begin, end, _ = sd.row_shard(num_rows, rank, world_size)
        nodes = perm[begin:end].clone()
        del perm
        all_reduce = None
        if world_size > 1:
            import torch.distributed as dist
            all_reduce = dist.all_reduce
        mean_ap, ap_se, ratio, r_se = _estimates((sum_ap, m, sum_a, sum_c), ap, dr.sum, dr.count, num_rows, n_nodes,
                                                 with_neighbours, all_reduce)
    return Estimate(mean_ap=mean_ap, mean_ap_se=ap_se, average_distortion=ratio, average_distortion_se=r_se,
                    sampled_worst_case_distortion=worst_case(hi, lo) if sum_c else math.nan, nodes=nodes, ap=ap,
                    distortion=dr)


def _estimates(sums, ap, a, c, num_rows, num_nodes, with_neighbours, all_reduce=None):
    """(mAP, its SE, R, its SE) of the module docstring.  sums = (sum of AP, m, sum of a_u, sum of c_u) over all S
    sampled rows; ap, a, c: this rank's per-row values (tensors).  The squared deviations from the estimates are
    summed in a second pass over the rows, and over the ranks by all_reduce (in place, on a tensor) when given."""
    sum_ap, m, sum_a, sum_c = sums
    m = int(m)
    mean_ap = sum_ap / m if m else math.nan
    ratio = sum_a / sum_c if sum_c else math.nan
    valid = ~torch.isnan(ap)
    dev_sq = torch.stack(((ap[valid] - mean_ap).square().sum(), (a - ratio * c.to(torch.float64)).square().sum()))
    if all_reduce is not None:
        all_reduce(dev_sq)
    ss_ap, ss_r = dev_sq.tolist()
    if m == with_neighbours:
        ap_se = 0.0
    elif m < 2:
        ap_se = math.nan
    else:
        ap_se = math.sqrt(ss_ap / (m - 1) / m * (1.0 - m / with_neighbours))
    if num_rows == num_nodes:
        r_se = 0.0 if sum_c else math.nan
    elif num_rows < 2 or not sum_c:
        r_se = math.nan
    else:
        c_bar = sum_c / num_rows
        r_se = math.sqrt((1.0 - num_rows / num_nodes) * ss_r / ((num_rows - 1) * num_rows * c_bar * c_bar))
    return mean_ap, ap_se, ratio, r_se


def worst_case(max_ratio, min_ratio):
    """worst-case distortion max(s d / g) / min(s d / g); inf when two distinct nodes share a point"""
    return max_ratio / min_ratio if min_ratio > 0 else math.inf


class MeanAveragePrecisionMetric:
    """The reference's metric call shape, `calculate_metric(distance_matrix)` on the whole (N, N) matrix
    (what Model.build_distance_matrix returns), computed on the device.

    The constructor differs from the reference's (whose source is not available): it takes the graph as the
    CSR adjacency `adj = (ptr, idx)` of graphs.adjacency_csr.  A numpy matrix is moved to the current CUDA
    device.  For graphs whose matrix does not fit, use mean_average_precision, which never holds it."""

    def __init__(self, adj):
        self.adj = adj

    def average_precision(self, distance_matrix):
        """(N,) float64 per-node AP on the matrix's device, NaN for a node without neighbours"""
        m = torch.as_tensor(distance_matrix, dtype=torch.float64)
        if not m.is_cuda:
            m = m.to(torch.device("cuda", torch.cuda.current_device()))
        m = m.detach().contiguous()
        ap = ops.average_precision(m, 0, _adjacency_on(self.adj, m.device))
        ops.check_status(m.device)
        return ap

    def calculate_metric(self, distance_matrix):
        """mAP: the mean of AP over the nodes with at least one neighbour"""
        ap = self.average_precision(distance_matrix)
        valid = ~torch.isnan(ap)
        return float(ap[valid].sum().item() / max(int(valid.sum().item()), 1))
