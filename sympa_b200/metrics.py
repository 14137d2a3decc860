"""Graph-reconstruction mean average precision on the device.

The reference evaluates by building the whole N x N distance matrix (Runner.evaluate, sympa/runner.py:124-154)
and handing it to MeanAveragePrecisionMetric (sympa/metrics.py), which ranks every row on the host.  Here the
matrix is streamed: rows are computed in blocks (sympa_dist_matrix) and each block is reduced to per-node average
precision on the device (sympa_average_precision) before the next block overwrites it, so memory is bounded by
the block, not by 8 N^2 bytes.

Definition (restated - the reference's metric code is not available, so parity with it is UNPINNED), with N(u)
the graph neighbours of u and d the manifold distance:

    AP(u) = 1/|N(u)| sum_{v in N(u)} |{v' in N(u) : d(u,v') <= d(u,v)}| / |{w != u : d(u,w) <= d(u,v)}|
    mAP   = mean of AP(u) over the nodes with |N(u)| > 0

Without ties this is what the usual argsort loop computes (sort the row, skip the node, record hits / i at the
i-th hit); with ties it is the "tied nodes rank first" value.  It does not depend on the model scale.
"""
import torch

from . import distributed as sd
from . import _lib, ops


def _adjacency_on(adj, device):
    ptr, idx = adj
    return (torch.as_tensor(ptr, dtype=torch.int64).to(device).contiguous(),
            torch.as_tensor(idx, dtype=torch.int64).to(device).contiguous())


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
    if not isinstance(table, torch.Tensor) or not table.is_cuda:
        raise RuntimeError("sympa_b200: mean_average_precision needs a CUDA table (there is no CPU path)")
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
        block = max(1, min(block_bytes // (8 * max(n_nodes, 1)), max(count_rows, 1)))
        buf = torch.empty(block * n_nodes, dtype=torch.float64, device=dev)
        ap = torch.empty(count_rows, dtype=torch.float64, device=dev)
        for r0 in range(begin, end, block):
            rc = min(block, end - r0)
            d = buf[: rc * n_nodes].view(rc, n_nodes)
            ops.dist_matrix(kind, metric, src, r0, rc, wsum, out=d)
            ops.average_precision(d, r0, adj, out=ap[r0 - begin: r0 - begin + rc])
        valid = ~torch.isnan(ap)
        totals = torch.stack((ap[valid].sum(), valid.sum().to(torch.float64)))
        if world_size > 1:
            import torch.distributed as dist
            dist.all_reduce(totals)
        ops.check_status(dev)
        sum_ap, count = totals.tolist()
    return sum_ap, int(count), ap


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
