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
"""
import collections
import math

import torch

from . import distributed as sd
from . import _lib, ops

Evaluation = collections.namedtuple("Evaluation", "average_distortion worst_case_distortion mean_ap ap distortion")
Evaluation.__doc__ = """Result of evaluate(): the two distortion figures and mAP (global when world_size > 1), the (rows,)
per-node AP of this rank's rows (NaN for a node without neighbours) and their per-node ops.DistortionRows."""


def _adjacency_on(adj, device):
    ptr, idx = adj
    return (torch.as_tensor(ptr, dtype=torch.int64).to(device).contiguous(),
            torch.as_tensor(idx, dtype=torch.int64).to(device).contiguous())


def _row_pass(who, manifold, table, adj, rows, block_bytes, world_size, rank, want_ap, scale):
    """The one streaming pass over row blocks of the distance matrix behind every metric here.  Per block:
    dist_matrix, then average_precision (want_ap) and hop_distances + distortion_rows (scale is not None) on that
    same block.  A block holds max(1, block_bytes // (bytes per entry * N)) rows, 8 bytes per entry (distances)
    plus 4 with distortion (hop distances).  Returns (sums, extremes, ap, distortion): sums = [sum_ap, count_ap]
    and / or [sum_delta, pairs] and extremes = (max, min) of s d / g, global when world_size > 1 (one SUM
    all-reduce, one MAX and one MIN), the per-node AP and DistortionRows of this rank's rows."""
    if not isinstance(table, torch.Tensor) or not table.is_cuda:
        raise RuntimeError(f"sympa_b200: {who} needs a CUDA table (there is no CPU path)")
    table = table.detach()
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
    kind = manifold.kind
    metric = "riem" if kind == "spd" else manifold.metric.name
    wsum = None if kind == "spd" else manifold._wsum(table)
    with torch.cuda.device(dev):
        src = table
        if kind == "bounded":
            t = ops._require(table, "table")
            ops._check_n(t.shape[-1])
            src = torch.empty_like(t)
            _lib.check(_lib.load().sympa_bounded_rows_to_upper(t.shape[-1], n_nodes, ops._ptr(t), ops._ptr(src),
                                                               ops._ptr(ops.status_word(dev)), ops._stream()))
            kind = "upper"
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
                ops.distortion_rows(d, h, r0, scale, out=ops.DistortionRows(*(o[part] for o in dr)))
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
