/* sympa_b200 - C ABI of the B200-native Siegel / SPD pair-distance hot path.
 *
 * Drop-in boundary for the one hot path of fedelopez77/sympa: everything the reference does
 * between `Model.forward` gathering two embedding rows and the embedding gradient being ready
 * for the optimizer.  All pointers are DEVICE pointers (caller allocates everything, the library
 * never allocates, frees or retains a pointer past the call), `stream` is a cudaStream_t passed as
 * void*, every call is asynchronous on that stream and returns an int status (0 = ok) for argument
 * errors only; numerical domain problems are OR-ed into the caller's device `status` word
 * (SYMPA_STATUS_* bits) instead of the reference's host-synchronising asserts
 * (sympa/manifolds/siegel_manifold.py:65-66).
 *
 * Layouts (sympa/math/csym_math.py:1-8, sympa/embeddings.py:59-68):
 *   complex symmetric point  (2, n, n) float64, [0] real part, [1] imaginary part, row-major
 *   spd point                (n, n)    float64
 *   table                    (num_rows, 2, n, n) / (num_rows, n, n), contiguous
 *   idx                      (num_pairs, 2) int64: (src row, dst row)   (train.py:95)
 *   vvd                      (num_pairs, n) ascending vector-valued distance
 *
 * The reference-side binding is a ctypes stub - see INTEGRATION.md.
 */
#ifndef SYMPA_B200_H_
#define SYMPA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 3: v2 plus additive entry points (sympa_dist_matrix, sympa_dist_backward_table, sympa_table_grad_scatter /
 *    _expand, sympa_rsgd_step_ex, sympa_distortion_loss_forward / _backward) and the bounded domain in
 *    sympa_rsgd_step; the saved state of the register-kernel sizes became packed (its size still comes from
 *    sympa_workspace_bytes, its layout was never part of the interface).
 * 4: the saved state is packed for EVERY matrix size (so sympa_backward_workspace_bytes is non-zero and
 *    sympa_table_grad_scatter / _expand work for all of them); the packed scatter runs in L2-sized passes
 *    (SYMPA_OPT_SCATTER_PASS_MB); sympa_rsgd_step takes the bounded-domain gradient unsymmetrised.
 *    Additive since: sympa_average_precision / _workspace_bytes (graph-reconstruction mAP over row blocks of
 *    the distance matrix); sympa_hop_distances / _workspace_bytes and sympa_distortion_rows (graph hop
 *    distances by breadth-first search, graph-reconstruction distortion over the same row blocks);
 *    sympa_sample_pairs / _workspace_bytes and SYMPA_STATUS_NO_PAIR (training pairs and their hop distances
 *    sampled by breadth-first search from a list of sources).  Callers
 *    that need them look the symbols up; the number stays 4 because nothing that a version-4 caller relies on
 *    changed. */
#define SYMPA_ABI_VERSION 4

/* manifold kinds: sympa/embeddings.py:144-149 ("upper", "bounded") and :142 ("spd") */
enum { SYMPA_KIND_UPPER = 0, SYMPA_KIND_BOUNDED = 1, SYMPA_KIND_SPD = 2 };
/* sympa/manifolds/metrics.py:6-12 */
enum { SYMPA_METRIC_RIEM = 0, SYMPA_METRIC_FONE = 1, SYMPA_METRIC_FINF = 2, SYMPA_METRIC_FMIN = 3, SYMPA_METRIC_WSUM = 4 };

/* return codes */
enum {
  SYMPA_OK = 0,
  SYMPA_ERR_BAD_ARG = 1,      /* null / inconsistent pointers, negative sizes */
  SYMPA_ERR_UNSUPPORTED = 2,  /* n outside [1, SYMPA_MAX_N], unknown kind / metric */
  SYMPA_ERR_CUDA = 3          /* launch failed; see sympa_last_cuda_error() */
};
#define SYMPA_MAX_N 10

/* bits of the device status word */
#define SYMPA_STATUS_NOT_PD 1u            /* a point is outside the manifold (Cholesky pivot <= 0) */
#define SYMPA_STATUS_TAKAGI_ABOVE_ONE 2u  /* siegel_manifold.py:66 assert */
#define SYMPA_STATUS_NO_CONVERGE 4u       /* Jacobi sweep cap reached */
#define SYMPA_STATUS_NON_FINITE 8u
#define SYMPA_STATUS_BAD_INDEX 16u        /* idx outside [0, num_rows) - the pair is skipped */
#define SYMPA_STATUS_NO_PAIR 32u          /* a sampling source reaches no other node (sympa_sample_pairs) */

int sympa_version(void);
const char* sympa_error_string(int code);
const char* sympa_last_cuda_error(void);

/* bytes of `saved_state` that sympa_dist_forward needs to make a later sympa_dist_backward possible:
 * the per-pair unit gradients d dist / d z1, d dist / d z2, i.e. 2 * num_pairs * point_doubles * 8. */
int64_t sympa_workspace_bytes(int kind, int n, int64_t num_pairs);

/* bytes of optional `scratch` (device memory, contents irrelevant, may be reused by the next call on
 * the same stream) that lets sympa_dist_forward / sympa_distortion_step run the larger matrix sizes
 * (upper half space, n > 4) as three kernels with the per-pair state parked in scratch instead of
 * shared memory.  0 when the configuration does not use scratch (always, unless the split path is
 * switched on with sympa_set_option).  Passing scratch == NULL (or fewer bytes) is always valid:
 * the single-kernel path is used. */
int64_t sympa_scratch_bytes(int kind, int n, int64_t num_pairs);

/* Riemannian SGD step on the whole table in one launch (SURVEY.md 8(f) rank 1): replaces
 * geoopt.optim.RiemannianSGD.step for the matrix table - egrad2rgrad (sympa/manifolds/upper_half.py:25-40),
 * retr (siegel_manifold.py:74-87) and projx (upper_half.py:42-66, csym_math.py:252-278) fused per row:
 *   upper:  X <- X - lr Y GX Y,  Y <- clamp_eig(Y - lr Y GY Y, eps) only when an eigenvalue is <= eps
 *   bounded: Z <- sym(Z - lr A G A), A = I - conj(Z) Z (bounded_domain.py:41-53), then the Takagi values
 *           above 1 - eps clamped to 1 - eps, only for the rows that have one (bounded_domain.py:55-84;
 *           what the reference's tests describe - the shipped projx crashes, SURVEY.md F3)
 *   spd:    X <- sym(X + U + U X^-1 U / 2),  U = -lr X sym(G) X        (geoopt, parity unpinned)
 * Rows whose gradient is identically zero are not touched (equivalent to the dense step, which leaves
 * them bit-identical).  lr_scale: optional device scalar multiplying lr (a clipping coefficient);
 * projected: optional device counter incremented by the number of rows the projection moved. */
int sympa_rsgd_step(int kind, int n, int64_t num_rows, double* table, const double* grad, double lr,
                    const double* lr_scale, unsigned long long* projected, void* stream);
/* The same with optimizer.zero_grad() (runner.py:117-118) fused in: zero_grad != 0 zeroes the gradient rows
 * that were applied (rows that were already zero are not touched), so that a training step on the fused
 * path is two launches: sympa_distortion_step and this. */
int sympa_rsgd_step_ex(int kind, int n, int64_t num_rows, double* table, double* grad, double lr,
                       const double* lr_scale, unsigned long long* projected, int zero_grad, void* stream);

/* process-wide tuning switches (host side only).  SYMPA_OPT_SPLIT_PATH: 0 (default) = larger matrix
 * sizes run as ONE cooperative kernel; 1 = three kernels through `scratch` (sympa_scratch_bytes then
 * reports a non-zero size).  Results are bit-identical either way. */
#define SYMPA_OPT_SPLIT_PATH 1
/* SYMPA_OPT_SCATTER_PASS_MB: megabytes of packed gradient table one pass of the table-gradient scatter covers
 * (default: unlimited = one pass; passes over L2-sized row ranges measured slower on the B200, see
 * sympa_b200.cu - kept for experiments). */
#define SYMPA_OPT_SCATTER_PASS_MB 2
int sympa_set_option(int option, int value);

/* Diagnostic: launches a pure FP64 FMA kernel (8 independent chains per thread, 8 CTAs of 256 threads
 * per SM, `iters` FMAs per chain) on `stream` and returns the number of floating-point operations it
 * issues (-1 on error); time it with events to get the device's attainable FP64 rate, the roofline
 * denominator bench.py reports for this FP64-pipe-bound path.  `out`: one device double (not written). */
int64_t sympa_probe_fp64(int iters, double* out, void* stream);

/* Forward of manifold.dist (siegel_manifold.py:41-72, bounded_domain.py:27-39, geoopt spd dist).
 * Operands come either materialised (z1, z2: (num_pairs, point)) or as a fused gather
 * (table + idx; replaces Embeddings.forward, sympa/embeddings.py:29-34).  Exactly one of the two
 * forms must be given.  wsum_w: n doubles (metrics.py:108) when metric == WSUM.
 * dist_out (num_pairs) is required; vvd_out (num_pairs, n) and status are optional.
 * saved_state == NULL -> forward only (evaluation, runner.py:124-154). */
int sympa_dist_forward(int kind, int n, int metric, int64_t num_pairs,
                       const double* z1, const double* z2,
                       const double* table, int64_t num_rows, const int64_t* idx,
                       const double* wsum_w,
                       double* dist_out, double* vvd_out, double* saved_state,
                       double* scratch, int64_t scratch_bytes,
                       unsigned int* status, void* stream);

/* All-pairs evaluation (SURVEY.md 8(f) rank 3): rows [row_begin, row_begin + row_count) of the
 * (num_rows x num_rows) matrix of manifold distances between the points of `table`, written row-major
 * into dist_out (row_count x num_rows) with exact zeros on the diagonal.  Replaces
 * Runner.build_distance_matrix (sympa/runner.py:142-154: num_rows forward calls of batch num_rows,
 * the diagonal entry asked for a neighbour and then overwritten with 0) by forward launches over
 * chunks of workspace_pairs pairs whose index pairs are generated on the device into idx_workspace
 * (2 * workspace_pairs int64, caller-allocated, contents irrelevant).  Forward only. */
int sympa_dist_matrix(int kind, int n, int metric, const double* table, int64_t num_rows,
                      int64_t row_begin, int64_t row_count, const double* wsum_w, double* dist_out,
                      int64_t* idx_workspace, int64_t workspace_pairs, unsigned int* status, void* stream);

/* Graph-reconstruction average precision of rows of a distance matrix (the mAP of the reference's evaluation;
 * its metric code is not available, so parity with it is unpinned - the definition is restated):
 *   AP(u) = 1/|N(u)| sum_{v in N(u)} |{v' in N(u) : d(u,v') <= d(u,v)}| / |{w != u : d(u,w) <= d(u,v)}|
 * which, without ties, is what an argsort-and-scan loop over the row computes (tied nodes rank first).
 * dist: row-major (row_count x num_cols) block holding rows [row_begin, row_begin + row_count) of the matrix -
 * what sympa_dist_matrix writes; column row_begin + r (the node itself) is never read as a candidate.
 * adj_ptr (num_cols + 1) / adj_idx: CSR adjacency of all num_cols nodes, rows free of duplicates; entries equal
 * to the row's node are ignored, entries outside [0, num_cols) are ignored and set SYMPA_STATUS_BAD_INDEX.
 * ap_out[r] = AP(row_begin + r), NaN for a row without neighbours or with a NaN distance (which also sets
 * SYMPA_STATUS_NON_FINITE).  A row's value is bit-identical whatever block, offset or launch shape it comes in.
 * workspace: device memory, contents irrelevant, of sympa_average_precision_workspace_bytes(row_count,
 * adj_entries) bytes where adj_entries >= adj_ptr[row_begin + row_count] - adj_ptr[row_begin] (the total entry
 * count always does); rows whose entries do not fit set SYMPA_STATUS_BAD_INDEX and get NaN. */
int64_t sympa_average_precision_workspace_bytes(int64_t row_count, int64_t adj_entries);
int sympa_average_precision(int64_t row_begin, int64_t row_count, int64_t num_cols, const double* dist,
                            const int64_t* adj_ptr, const int64_t* adj_idx, double* ap_out,
                            void* workspace, int64_t workspace_bytes, unsigned int* status, void* stream);

/* Hop distances of the undirected graph given by the CSR adjacency adj_ptr (num_nodes + 1) / adj_idx (valid
 * pointers: non-decreasing, every entry of [adj_ptr[0], adj_ptr[num_nodes]) readable), by breadth-first search
 * from every source of rows [row_begin, row_begin + row_count).  hops_out: row-major (row_count x num_nodes)
 * int32, entry [r][v] = hop distance from row_begin + r to v, 0 on the diagonal, -1 where v is unreachable.
 * Entries outside [0, num_nodes) are skipped and set SYMPA_STATUS_BAD_INDEX.  The output is identical on every
 * run and for every block or offset (breadth-first distances are unique; only the queue order varies).
 * workspace: device memory, contents irrelevant, of sympa_hop_distances_workspace_bytes(num_nodes) bytes - one
 * queue of num_nodes int32 per resident CTA of a persistent grid, so it does not grow with row_count.  Work per
 * source is O(num_nodes + entries) with one CTA barrier per BFS level. */
int64_t sympa_hop_distances_workspace_bytes(int64_t num_nodes);
int sympa_hop_distances(int64_t row_begin, int64_t row_count, int64_t num_nodes, const int64_t* adj_ptr,
                        const int64_t* adj_idx, int32_t* hops_out, void* workspace, int64_t workspace_bytes,
                        unsigned int* status, void* stream);

/* Training pairs sampled from the undirected graph of the CSR adjacency adj_ptr (num_nodes + 1) / adj_idx (as for
 * sympa_hop_distances), K = pairs_per_source per source, without an N-wide row per source ever reaching the output.
 * With mix the SplitMix64 finalizer (all arithmetic mod 2^64)
 *   mix(x):  x += 0x9E3779B97F4A7C15;  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9;
 *            x = (x ^ (x >> 27)) * 0x94D049BB133111EB;  x ^= x >> 31
 *   h(seed, epoch, tag, a, b) = mix(mix(mix(mix(mix(seed) ^ epoch) ^ tag) ^ a) ^ b)
 * and R(u) the nodes reachable from u, c = |R(u)| - 1: draw k = 0 .. K-1 of source u is the r-th node (0-based) of
 * R(u) \ {u} in ascending node id, r = floor(h(seed, epoch, 0, u, k) * c / 2^64), with its hop distance g >= 1.
 * Draws are uniform with replacement (bias at most c / 2^64) and depend on nothing else: not the queue order, the
 * launch shape, the source's position in the list or the other sources.
 * sources: num_sources int64 node ids.  idx_out: (num_sources * K, 2) int64 [u, dst]; dist_out: (num_sources * K)
 * float64 g; the pairs of sources[i] are rows i*K .. i*K + K-1, k ascending.  A source outside [0, num_nodes) sets
 * SYMPA_STATUS_BAD_INDEX, one that reaches no other node SYMPA_STATUS_NO_PAIR; both get K pairs (u, u) at distance
 * 0.  Adjacency entries outside [0, num_nodes) are skipped and set SYMPA_STATUS_BAD_INDEX.
 * workspace: device memory, contents irrelevant, of sympa_sample_pairs_workspace_bytes(num_nodes) bytes - per
 * resident CTA of a persistent grid a queue, a row of hop distances and the reached set with its popcount prefixes,
 * about 8.25 bytes per node; it grows with neither num_sources nor K.  Work per source is one breadth-first search
 * (O(num_nodes + entries)) plus O(K log num_nodes). */
int64_t sympa_sample_pairs_workspace_bytes(int64_t num_nodes);
int sympa_sample_pairs(int64_t num_nodes, const int64_t* adj_ptr, const int64_t* adj_idx, int64_t num_sources,
                       const int64_t* sources, int64_t pairs_per_source, uint64_t seed, uint64_t epoch,
                       int64_t* idx_out, double* dist_out, void* workspace, int64_t workspace_bytes,
                       unsigned int* status, void* stream);

/* Graph-reconstruction distortion of rows of a distance matrix (the reference's evaluation reports the average;
 * its metric code is not available, so parity with it is unpinned - the definition is restated).  With g(u, w)
 * the hop distance, s the model scale and d(u, w) row u, column w of the distance matrix, over the pairs u < w
 * connected in the graph (the reference's triplets):
 *   delta(u, w) = |s d(u, w) - g(u, w)| / g(u, w)
 *   average distortion    = mean of delta over all pairs
 *   worst-case distortion = max(s d / g) / min(s d / g) over all pairs
 * dist: the (row_count x num_cols) float64 block of rows [row_begin, row_begin + row_count) (sympa_dist_matrix),
 * hops: the int32 block of the same rows (sympa_hop_distances).  For row u = row_begin + r, over the columns
 * w > u with hops >= 1: sum_out[r] = sum of delta, count_out[r] = the number of pairs, max_out[r] / min_out[r] =
 * the extremes of s d / g (-inf / +inf for a row without pairs).  A NaN among the row's scaled distances makes
 * all three float outputs NaN and sets SYMPA_STATUS_NON_FINITE.  Each row is summed in one fixed order: its
 * values are bit-identical whatever block, offset or shard it comes in.  Reads 12 bytes per entry of the
 * row's upper part. */
int sympa_distortion_rows(int64_t row_begin, int64_t row_count, int64_t num_cols, const double* dist, const int32_t* hops,
                          double scale, double* sum_out, int64_t* count_out, double* max_out, double* min_out,
                          unsigned int* status, void* stream);

/* Backward: replaces autograd through the ~250 torch ops of dist plus the gather backward.
 * grad_dist (num_pairs) is dL/d dist.  Materialised form: grad_z1 / grad_z2 are OVERWRITTEN with
 * the (symmetric) gradients.  Table form: grad_table (num_rows, point) is ACCUMULATED into with
 * FP64 atomics (caller zeroes it, as zero_grad does at runner.py:95-96).  For metric WSUM pass vvd
 * and wsum_w to have dL/dw accumulated into grad_wsum_w (n doubles). */
int sympa_dist_backward(int kind, int n, int metric, int64_t num_pairs,
                        const double* grad_dist, const double* saved_state,
                        double* grad_z1, double* grad_z2,
                        double* grad_table, int64_t num_rows, const int64_t* idx,
                        const double* vvd, const double* wsum_w, double* grad_wsum_w,
                        void* stream);

/* Table-gradient backward with an optional workspace (same result as sympa_dist_backward in its table
 * form).  workspace: sympa_backward_workspace_bytes(kind, n, num_rows) bytes of device memory (contents
 * irrelevant; 0 = this configuration does not use one).  When given and the batch covers the table
 * densely (2 * num_pairs >= num_rows) the scatter-add runs on a packed (lower-triangle) gradient table in
 * the workspace and the dense symmetric rows are produced in one pass at the end; otherwise the direct
 * scatter is used.  overwrite != 0: grad_table is WRITTEN (the caller need not zero it - what an autograd
 * backward wants for its freshly allocated gradient); overwrite == 0: accumulated into, as above. */
int64_t sympa_backward_workspace_bytes(int kind, int n, int64_t num_rows);
int sympa_dist_backward_table(int kind, int n, int metric, int64_t num_pairs,
                              const double* grad_dist, const double* saved_state,
                              double* grad_table, int64_t num_rows, const int64_t* idx,
                              const double* vvd, const double* wsum_w, double* grad_wsum_w,
                              double* workspace, int64_t workspace_bytes, int overwrite, void* stream);

/* The two halves of the packed route of sympa_dist_backward_table as separate calls, so that a data-parallel
 * caller can all-reduce the PACKED gradient table (62 % of the dense bytes at n = 4) between them - the one
 * collective of the path (DDP's all-reduce of the dense table gradient, train.py:59):
 *   sympa_table_grad_scatter   workspace <- 0, then scatter-add of grad_dist * unit gradients (packed rows);
 *                              also dL/dw of the wsum metric when grad_wsum_w is given
 *   [ncclAllReduce over workspace, sympa_backward_workspace_bytes(kind, n, num_rows) bytes of doubles]
 *   sympa_table_grad_expand    grad_table <- (or +=) the dense symmetric rows
 * (Every configuration has a packed workspace since ABI 4.) */
int sympa_table_grad_scatter(int kind, int n, int metric, int64_t num_pairs,
                             const double* grad_dist, const double* saved_state,
                             int64_t num_rows, const int64_t* idx,
                             const double* vvd, const double* wsum_w, double* grad_wsum_w,
                             double* workspace, int64_t workspace_bytes, void* stream);
int sympa_table_grad_expand(int kind, int n, int64_t num_rows, const double* workspace, double* grad_table,
                            int overwrite, void* stream);
/* The scatter half WITHOUT the zeroing: adds the batch's contributions to a packed gradient table the caller keeps
 * across several batches of one step (gradient accumulation, runner.py:104: grad_accum_steps) - the caller zeroes the
 * workspace at the start of the step, calls this once per batch, then [all-reduces and] expands once per step.
 * (dL/dw of the wsum metric: sympa_dist_backward with only grad_wsum_w.)
 * max_sms > 0 with tickets != NULL (8 bytes of device memory, contents irrelevant, owned by the call until it has
 * run): the scatter confines itself to the SMs with id < max_sms, so that a caller who issues it on a side stream
 * leaves the other SMs to the forward kernel of the next batch (the two kernels cannot share an SM); max_sms = 0:
 * the whole GPU. */
int sympa_table_grad_scatter_add(int kind, int n, int64_t num_pairs, const double* grad_dist, const double* saved_state,
                                 int64_t num_rows, const int64_t* idx, double* workspace, int64_t workspace_bytes,
                                 int max_sms, unsigned int* tickets, void* stream);
/* The scatter half restricted to the destination rows [row_begin, row_end): zeroes that range of the packed
 * workspace and scatter-adds the batch's contributions to it (dL/dw of the wsum metric is NOT computed here:
 * use sympa_dist_backward with only grad_wsum_w).  Lets a data-parallel caller pipeline the collective: scatter
 * range k, start the all-reduce of range k on a side stream, scatter range k + 1 meanwhile - the all-reduce of
 * DDP's dense table gradient (train.py:59) disappears behind the scatter.  num_pairs == 0 only zeroes. */
int sympa_table_grad_scatter_rows(int kind, int n, int64_t num_pairs, const double* grad_dist, const double* saved_state,
                                  int64_t num_rows, const int64_t* idx, int64_t row_begin, int64_t row_end,
                                  double* workspace, int64_t workspace_bytes, void* stream);

/* Bounded domain by rows.  BoundedDomainManifold.dist (bounded_domain.py:27-39) maps both operands to the upper
 * half space with the inverse Cayley transform and calls the upper-half dist.  The transform acts on points,
 * so on the table path it can be applied ONCE PER TABLE ROW instead of once per pair and operand:
 *   sympa_bounded_rows_to_upper   upper_out[r] = i (I + z_r)(I - z_r)^-1      (num_rows, 2, n, n)
 *   ... sympa_dist_forward / backward with SYMPA_KIND_UPPER on upper_out ...
 *   sympa_bounded_rows_backward   grad_table[r] (=, +=) conj(N_r) (2 G_Y - 2i G_X) conj(N_r),  N_r = (I - z_r)^-1,
 *                                 G = grad_upper[r] the (symmetric) upper-half gradient of the row
 * Worth it when the batch covers the table densely; the per-pair bounded kernels remain for materialised
 * operands and sparse batches. */
int sympa_bounded_rows_to_upper(int n, int64_t num_rows, const double* table, double* upper_out,
                                unsigned int* status, void* stream);
int sympa_bounded_rows_backward(int n, int64_t num_rows, const double* table, const double* grad_upper,
                                double* grad_table, int overwrite, void* stream);

/* Embeddings.check_all_points (sympa/embeddings.py:41-47: a Python loop over the points calling
 * check_point_on_manifold, run once per epoch at runner.py:91) as one launch over the table: every n x n block
 * allclose to its transpose (atol, rtol: siegel_manifold.py:123-124), then upper: det(Im z) > 0
 * (upper_half.py:93-114); bounded: I - conj(z) z allclose to its conjugate transpose (bounded_domain.py:119-150);
 * spd: eigenvalues > -atol (geoopt).  *result (8 bytes of device memory, written by the call) = ~0 when every row
 * passes, else (first offending row << 8) | reason, reason 1 = not symmetric, 2 = the kind's predicate. */
#define SYMPA_CHECK_OK 0xFFFFFFFFFFFFFFFFull
int sympa_check_points(int kind, int n, int64_t num_rows, const double* table, double atol, double rtol,
                       unsigned long long* result, void* stream);

/* AverageDistortionLoss.calculate_loss (sympa/losses.py:10-19): loss_out (1 double, ACCUMULATED into) +=
 * sum_p |(manifold_dist_p / graph_dist_p)^2 - 1|, and its backward grad_manifold_dist_p = grad_loss *
 * sign(.) * 2 manifold_dist_p / graph_dist_p^2 (grad_loss: 1 device double) - one kernel each instead of the
 * ~11 element-wise torch kernels of the Python expression (5 % of a step at n = 4). */
int sympa_distortion_loss_forward(int64_t num_pairs, const double* graph_dist, const double* manifold_dist,
                                  double* loss_out, void* stream);
int sympa_distortion_loss_backward(int64_t num_pairs, const double* graph_dist, const double* manifold_dist,
                                   const double* grad_loss, double* grad_manifold_dist, void* stream);

/* One fused launch for a training step of the distortion objective (sympa/losses.py:16-19 with
 * the scale of sympa/model.py:30):   L = sum_p | (scale * dist_p / graph_dist_p)^2 - 1 |.
 * Gathers both rows, computes dist, the loss term and its derivative, and scatter-adds
 * dL/d table into grad_table.  loss_out, grad_scale (1 double each), grad_wsum_w (n) and grad_table
 * are ACCUMULATED into; dist_out (num_pairs) is optional. */
int sympa_distortion_step(int kind, int n, int metric, int64_t num_pairs,
                          const double* table, int64_t num_rows, const int64_t* idx,
                          const double* graph_dist, double scale, const double* wsum_w,
                          double* grad_table, double* grad_wsum_w, double* grad_scale, double* loss_out,
                          double* dist_out, double* scratch, int64_t scratch_bytes,
                          unsigned int* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SYMPA_B200_H_ */
