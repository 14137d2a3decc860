// Graph hop distances and graph-reconstruction distortion of rows of a distance matrix
// (sympa_hop_distances, sympa_distortion_rows).
//
//   hop_bfs_kernel         persistent grid, one CTA per source row at a time (rows pulled as tickets from a
//                          counter at the head of the workspace): level-synchronous breadth-first search whose
//                          queue is the CTA's own slice of the workspace; a vertex is claimed with one atomic on
//                          the visited set - a bitmap in shared memory up to SY_HOP_SMEM_VISITED_BYTES, the
//                          output row itself (-1 = not reached yet, atomicCAS) beyond - so it enters the queue
//                          exactly once and its hop count is the level that claimed it - unique, whatever order
//                          the queue was filled in.  The bitmap halves the kernel's time on the workloads of
//                          profiles/eval_b200.py (B200: 7.6 -> 3.8 ms per block of the 2^17-node random tree,
//                          profiles/eval_hop_variants_b200.txt); 1 CTA per SM measured slower on every workload, 4
//                          faster on config 3 (0.77 against 1.27 ms) but slower on both trees
//   distortion_rows_kernel one CTA per row: over the columns w > u with a hop distance >= 1, the sum of
//                          |s d - g| / g, the pair count and the extremes of s d / g; every thread walks a fixed
//                          residue class of the row's columns and the partial results are combined by a fixed
//                          tree, so a row's values do not depend on the block it came in
#pragma once

#include <cooperative_groups.h>
#include <math.h>
#include <stdint.h>

namespace sympa {

#define SY_HOP_THREADS 512
#ifndef SY_HOP_CTAS_PER_SM            // -D overridable, for the variant builds of profiles/eval_hop_variants.py
#define SY_HOP_CTAS_PER_SM 2
#endif
#define SY_HOP_HEADER_BYTES 256       // the ticket counter, padded so that the queues stay aligned
// Graphs whose visited bitmap fits the default 48 KB dynamic + static shared-memory limit keep the visited set in
// shared memory; the 256 bytes left over cover the kernel's static shared memory (16 bytes), so no opt-in is needed.
// Up to 391 168 nodes.  0 = always the output row in global memory.
#ifndef SY_HOP_SMEM_VISITED_BYTES
#define SY_HOP_SMEM_VISITED_BYTES (48 * 1024 - 256)
#endif
#define SY_DISTORTION_THREADS 256

// Neighbour w of a frontier vertex, reached at level next_level: claims it and appends it to the next frontier
// (queue[tail + k], k from the shared counter, one atomicAdd per group of converged lanes).  SMEM_VISITED: the
// visited set is a bitmap in shared memory and the output entry is a plain store; otherwise the output row is
// the visited set and the claim an atomicCAS on it.
template <bool SMEM_VISITED>
__device__ __forceinline__ void hop_visit(int64_t w, int num_nodes, int* row, unsigned int* visited, int next_level,
                                          int* queue, int tail, int* next_count, unsigned int* status) {
  namespace cg = cooperative_groups;
  if (w < 0 || w >= num_nodes) {
    if (status) atomicOr(status, SYMPA_STATUS_BAD_INDEX);
    return;
  }
  if (SMEM_VISITED) {
    const unsigned int bit = 1u << (w & 31);
    volatile unsigned int* word = visited + (w >> 5);
    if (*word & bit) return;                              // already claimed: skip the atomic
    if (atomicOr(visited + (w >> 5), bit) & bit) return;
    row[w] = next_level;
  } else {
    if (__ldcg(row + w) != -1) return;
    if (atomicCAS(row + w, -1, next_level) != -1) return;
  }
  cg::coalesced_group g = cg::coalesced_threads();
  int base = 0;
  if (g.thread_rank() == 0) base = atomicAdd(next_count, (int)g.size());
  base = g.shfl(base, 0);
  queue[tail + base + (int)g.thread_rank()] = (int)w;
}

template <bool SMEM_VISITED>
__global__ void __launch_bounds__(SY_HOP_THREADS) hop_bfs_kernel(int64_t row_begin, int row_count, int num_nodes,
                                                                 const int64_t* __restrict__ adj_ptr,
                                                                 const int64_t* __restrict__ adj_idx,
                                                                 int* __restrict__ hops, int* __restrict__ queues,
                                                                 unsigned int* __restrict__ ticket,
                                                                 unsigned int* __restrict__ status) {
  __shared__ int s_row;
  // frontier sizes, rotating over three slots: at level L the current frontier's size is read from slot
  // (L + 2) % 3, the next one is counted in slot L % 3, and slot (L + 1) % 3 - last read at level L - 1 - is
  // cleared for level L + 1.  One barrier per level.
  __shared__ int s_count[3];
  extern __shared__ unsigned int s_visited[];           // SMEM_VISITED: (num_nodes + 31) / 32 words
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int nwarps = blockDim.x >> 5;
  int* queue = queues + (int64_t)blockIdx.x * num_nodes;
  for (;;) {
    if (threadIdx.x == 0) s_row = (int)atomicAdd(ticket, 1u);
    __syncthreads();
    const int r = s_row;
    if (r >= row_count) return;
    const int src = (int)(row_begin + r);
    int* row = hops + (int64_t)r * num_nodes;
    for (int v = threadIdx.x; v < num_nodes; v += blockDim.x) row[v] = v == src ? 0 : -1;
    if (SMEM_VISITED)
      for (int k = threadIdx.x; k < (num_nodes + 31) / 32; k += blockDim.x)
        s_visited[k] = k == src / 32 ? 1u << (src & 31) : 0u;
    if (threadIdx.x == 0) {
      queue[0] = src;
      s_count[0] = 0;
      s_count[1] = 0;
      s_count[2] = 1;
    }
    __syncthreads();
    int hi = 0;
    for (int level = 0;; ++level) {
      const int cnt = s_count[(level + 2) % 3];
      if (cnt == 0) break;
      const int lo = hi;
      hi = lo + cnt;
      int* next_count = s_count + level % 3;
      // 32 frontier vertices per warp; a vertex with >= 32 neighbours is expanded by the whole warp, the
      // others by their own lane
      for (int base = lo + warp * 32; base < hi; base += nwarps * 32) {
        const int i = base + lane;
        int64_t p0 = 0, p1 = 0;
        if (i < hi) {
          const int v = queue[i];
          p0 = __ldg(adj_ptr + v);
          p1 = __ldg(adj_ptr + v + 1);
        }
        const bool wide = p1 - p0 >= 32;
        unsigned todo = __ballot_sync(full, wide);
        while (todo) {
          const int l = __ffs(todo) - 1;
          todo &= todo - 1;
          const int64_t q0 = __shfl_sync(full, p0, l), q1 = __shfl_sync(full, p1, l);
          for (int64_t j = q0 + lane; j < q1; j += 32)
            hop_visit<SMEM_VISITED>(__ldg(adj_idx + j), num_nodes, row, s_visited, level + 1, queue, hi, next_count,
                                    status);
        }
        if (!wide)
          for (int64_t j = p0; j < p1; ++j)
            hop_visit<SMEM_VISITED>(__ldg(adj_idx + j), num_nodes, row, s_visited, level + 1, queue, hi, next_count,
                                    status);
      }
      if (threadIdx.x == 0) s_count[(level + 1) % 3] = 0;
      __syncthreads();
    }
  }
}

__global__ void __launch_bounds__(SY_DISTORTION_THREADS) distortion_rows_kernel(
    int64_t row_begin, int64_t num_cols, const double* __restrict__ dist, const int* __restrict__ hops, double scale,
    double* __restrict__ sum_out, int64_t* __restrict__ count_out, double* __restrict__ max_out,
    double* __restrict__ min_out, unsigned int* __restrict__ status) {
  constexpr int W = SY_DISTORTION_THREADS / 32;
  __shared__ double s_sum[W], s_max[W], s_min[W];
  __shared__ long long s_cnt[W];
  const int64_t r = blockIdx.x;
  const int64_t u = row_begin + r;
  const double* drow = dist + r * num_cols;
  const int* hrow = hops + r * num_cols;
  double sum = 0.0, hi = -INFINITY, lo = INFINITY;
  long long cnt = 0;
  int nan = 0;
  for (int64_t w = u + 1 + threadIdx.x; w < num_cols; w += SY_DISTORTION_THREADS) {
    const int g = __ldcs(hrow + w);
    const double d = __ldcs(drow + w);
    if (g < 1) continue;
    ++cnt;
    const double sd = scale * d;
    if (isnan(sd)) {
      nan = 1;
      continue;
    }
    const double gd = (double)g;
    sum += fabs(sd - gd) / gd;
    const double ratio = sd / gd;
    hi = fmax(hi, ratio);
    lo = fmin(lo, ratio);
  }
  for (int o = 16; o > 0; o >>= 1) {     // xor butterfly: a fixed order
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
    s_sum[warp] = sum;
    s_cnt[warp] = cnt;
    s_max[warp] = hi;
    s_min[warp] = lo;
  }
  nan = __syncthreads_or(nan);
  if (threadIdx.x != 0) return;
  for (int k = 1; k < W; ++k) {
    sum += s_sum[k];
    cnt += s_cnt[k];
    hi = fmax(hi, s_max[k]);
    lo = fmin(lo, s_min[k]);
  }
  if (nan) {
    sum = hi = lo = NAN;
    if (status) atomicOr(status, SYMPA_STATUS_NON_FINITE);
  }
  sum_out[r] = sum;
  count_out[r] = (int64_t)cnt;
  max_out[r] = hi;
  min_out[r] = lo;
}

}  // namespace sympa
