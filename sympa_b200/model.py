"""Mirror of sympa/model.py with the gather fused into the distance kernel."""
import torch
import torch.nn as nn

from .embeddings import ManifoldFactory, MatrixEmbeddings


class Model(nn.Module):
    """Graph embedding model (sympa/model.py:6-47).  `args` needs manifold, metric, dims, num_points,
    scale_init, scale_coef, train_scale."""

    def __init__(self, args):
        super().__init__()
        self.manifold = ManifoldFactory.get_manifold(args.manifold, args.metric, args.dims)
        self.embeddings = MatrixEmbeddings(args.num_points, args.dims, self.manifold)
        self.scale_coef = args.scale_coef
        self.scale = nn.Parameter(torch.tensor([self.scale_coef * args.scale_init], dtype=torch.float64),
                                  requires_grad=args.train_scale)

    def forward(self, input_triplet):
        """(b, >=2) int64 (src, dst, ...) -> (b,) scaled distances (model.py:16-30); one fused kernel
        instead of two gathers + dist."""
        idx = input_triplet[:, :2].contiguous()
        return self.manifold.dist_from_table(self.embeddings.embeds, idx) * self.get_scale()

    def distance(self, src_embeds, dst_embeds):   # model.py:32-38
        return self.manifold.dist(src_embeds, dst_embeds)

    def build_distance_matrix(self, rows_per_call=None):
        """(N, N) matrix of scaled manifold distances between all embeddings, zeros on the diagonal
        (Runner.build_distance_matrix, sympa/runner.py:142-154, which calls the model once per node):
        forward-only launches over chunks of pairs, indices generated on the device."""
        table = self.embeddings.embeds.detach()
        n_pts = table.shape[0]
        with torch.no_grad():
            if rows_per_call is None:
                return self.manifold.dist_matrix(table) * self.get_scale()
            out = torch.empty(n_pts, n_pts, dtype=torch.float64, device=table.device)
            for r0 in range(0, n_pts, rows_per_call):
                rc = min(rows_per_call, n_pts - r0)
                out[r0:r0 + rc] = self.manifold.dist_matrix(table, r0, rc) * self.get_scale()
            return out

    def mean_average_precision(self, adj, **kw):
        """Graph-reconstruction mAP of the embedding table against the CSR adjacency `adj`, streamed over row
        blocks of the distance matrix (see sympa_b200.metrics.mean_average_precision for the keywords)."""
        from .metrics import mean_average_precision
        sum_ap, count, _ = mean_average_precision(self.manifold, self.embeddings.embeds, adj, **kw)
        return sum_ap / max(count, 1)

    def average_distortion(self, adj, **kw):
        """Average graph-reconstruction distortion of the embedding table, distances scaled by get_scale(), against
        the hop distances of the CSR adjacency `adj`, streamed over row blocks of the distance matrix (see
        sympa_b200.metrics.average_distortion for the keywords)."""
        from .metrics import average_distortion
        total, count, _, _, _ = average_distortion(self.manifold, self.embeddings.embeds, adj, scale=self._eval_scale(), **kw)
        return total / count if count else float("nan")

    def evaluate(self, adj, **kw):
        """(average distortion, mAP) - the pair Runner.evaluate (sympa/runner.py:124-154) reports - in one pass over
        row blocks of the distance matrix (see sympa_b200.metrics.evaluate for the keywords)."""
        from .metrics import evaluate
        r = evaluate(self.manifold, self.embeddings.embeds, adj, scale=self._eval_scale(), **kw)
        return r.average_distortion, r.mean_ap

    def estimate(self, adj, num_rows, **kw):
        """mAP and average distortion, with standard errors, estimated from num_rows sampled rows of the distance
        matrix, distances scaled by get_scale(): the metrics.Estimate of sympa_b200.metrics.estimate (see there for
        the keywords)."""
        from .metrics import estimate
        return estimate(self.manifold, self.embeddings.embeds, adj, num_rows, scale=self._eval_scale(), **kw)

    def nearest(self, queries, k, **kw):
        """The k nearest nodes of every node in `queries` (1-D int64 ids), distances scaled by get_scale(): the
        metrics.Neighbours of sympa_b200.metrics.nearest (see there for the keywords)."""
        from .metrics import nearest
        return nearest(self.manifold, self.embeddings.embeds, queries, k, scale=self._eval_scale(), **kw)

    def link_prediction(self, pairs, filter_adj, **kw):
        """Filtered link-prediction ranks of the directed query pairs `pairs` ((E, 2) int64) against the CSR adjacency
        `filter_adj` of the known edges, with MRR and Hits@k: the metrics.LinkPrediction of
        sympa_b200.metrics.link_prediction (see there for the keywords).  Ranks do not depend on the scale."""
        from .metrics import link_prediction
        return link_prediction(self.manifold, self.embeddings.embeds, pairs, filter_adj, **kw)

    def _eval_scale(self):
        with torch.no_grad():
            return float(self.get_scale().item())

    def get_scale(self):   # model.py:40-41
        return (self.scale / self.scale_coef).clamp_min(0.1)

    def check_all_points(self):
        return self.embeddings.check_all_points()

    def embeds_norm(self):
        return self.embeddings.norm()
