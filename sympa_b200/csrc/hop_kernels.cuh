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
//   sample_pairs_kernel    persistent grid, one CTA per source at a time: the same breadth-first search (the shared
//                          level loop hop_bfs_levels) into the CTA's own queue and row, then K destinations drawn
//                          uniformly from the reached set by a binary search over per-word popcount prefixes of
//                          it; only the K pairs per source reach the output
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

// The level loop of one breadth-first search, shared by hop_bfs_kernel and sample_pairs_kernel.  On entry the source
// is claimed (its visited bit or row entry set), queue[0] holds it and s_count = {0, 0, 1}, all made visible by a
// barrier.  s_count holds the frontier sizes, rotating over three slots: at level L the current frontier's size is
// read from slot (L + 2) % 3, the next one is counted in slot L % 3, and slot (L + 1) % 3 - last read at level
// L - 1 - is cleared for level L + 1.  One barrier per level.  Returns, in every thread, the number of vertices
// claimed (the source included); queue[0, that number) holds them, row[v] is the hop distance of each.
template <bool SMEM_VISITED>
__device__ __forceinline__ int hop_bfs_levels(int num_nodes, const int64_t* __restrict__ adj_ptr,
                                              const int64_t* __restrict__ adj_idx, int* row, unsigned int* visited,
                                              int* queue, int* s_count, unsigned int* status) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int nwarps = blockDim.x >> 5;
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
          hop_visit<SMEM_VISITED>(__ldg(adj_idx + j), num_nodes, row, visited, level + 1, queue, hi, next_count,
                                  status);
      }
      if (!wide)
        for (int64_t j = p0; j < p1; ++j)
          hop_visit<SMEM_VISITED>(__ldg(adj_idx + j), num_nodes, row, visited, level + 1, queue, hi, next_count,
                                  status);
    }
    if (threadIdx.x == 0) s_count[(level + 1) % 3] = 0;
    __syncthreads();
  }
  return hi;
}

template <bool SMEM_VISITED>
__global__ void __launch_bounds__(SY_HOP_THREADS) hop_bfs_kernel(int64_t row_begin, int row_count, int num_nodes,
                                                                 const int64_t* __restrict__ adj_ptr,
                                                                 const int64_t* __restrict__ adj_idx,
                                                                 int* __restrict__ hops, int* __restrict__ queues,
                                                                 unsigned int* __restrict__ ticket,
                                                                 unsigned int* __restrict__ status) {
  __shared__ int s_row;
  __shared__ int s_count[3];
  extern __shared__ unsigned int s_visited[];           // SMEM_VISITED: (num_nodes + 31) / 32 words
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
    hop_bfs_levels<SMEM_VISITED>(num_nodes, adj_ptr, adj_idx, row, s_visited, queue, s_count, status);
  }
}

// SplitMix64 finalizer and the sampler's hash h(seed, epoch, tag, a, b) (sympa_sample_pairs in the header)
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__device__ __forceinline__ uint64_t sample_hash(uint64_t seed, uint64_t epoch, uint64_t tag, uint64_t a, uint64_t b) {
  return splitmix64(splitmix64(splitmix64(splitmix64(splitmix64(seed) ^ epoch) ^ tag) ^ a) ^ b);
}

// Position of the j-th (0-based) set bit of m; m has more than j set bits.
__device__ __forceinline__ int select_bit(unsigned m, int j) {
  int pos = 0;
#pragma unroll
  for (int width = 16; width > 0; width >>= 1) {
    const unsigned low = m & ((1u << width) - 1u);
    const int c = __popc(low);
    if (j >= c) {
      j -= c;
      m >>= width;
      pos += width;
    } else {
      m = low;
    }
  }
  return pos;
}

// Ints of one CTA's slice of the sampler's workspace: queue and row (num_nodes each), the reached set as a bitmap
// and its per-word exclusive popcount prefix ((num_nodes + 31) / 32 words each), rounded up to 16 bytes.
__host__ __device__ __forceinline__ int64_t sample_slice_ints(int64_t num_nodes) {
  return (2 * num_nodes + 2 * ((num_nodes + 31) / 32) + 3) / 4 * 4;
}

// Persistent grid, one CTA per source at a time (sources pulled as tickets): breadth-first search from the source
// (the level loop of hop_bfs_kernel, into the CTA's own queue and row), then the reached set minus the source as a
// bitmap (the shared-memory visited set itself, or built from the row), per-word popcount prefixes of it, and
// each of the K draws resolved by a binary search over the prefixes plus a select within the word.
template <bool SMEM_VISITED>
__global__ void __launch_bounds__(SY_HOP_THREADS, SY_HOP_CTAS_PER_SM) sample_pairs_kernel(
    int num_sources, int num_nodes, const int64_t* __restrict__ adj_ptr, const int64_t* __restrict__ adj_idx,
    const int64_t* __restrict__ sources, int64_t pairs_per_source, uint64_t seed, uint64_t epoch,
    int64_t* __restrict__ idx_out, double* __restrict__ dist_out, int* __restrict__ slices,
    unsigned int* __restrict__ ticket, unsigned int* __restrict__ status) {
  __shared__ unsigned int s_item;   // unsigned: the tickets past the last source stay above it (< 2^31 + grid)
  __shared__ int s_count[3];
  __shared__ int s_scan[SY_HOP_THREADS / 32];
  extern __shared__ unsigned int s_visited[];           // SMEM_VISITED: (num_nodes + 31) / 32 words
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int nwarps = blockDim.x >> 5;
  const int words = (num_nodes + 31) / 32;
  int* queue = slices + (int64_t)blockIdx.x * sample_slice_ints(num_nodes);
  int* row = queue + num_nodes;
  unsigned int* bits = SMEM_VISITED ? s_visited : reinterpret_cast<unsigned int*>(row + num_nodes);
  int* prefix = row + num_nodes + words;
  const int64_t K = pairs_per_source;
  for (;;) {
    __syncthreads();                                    // the previous source is done with s_item and the bitmap
    if (threadIdx.x == 0) s_item = atomicAdd(ticket, 1u);
    __syncthreads();
    const unsigned int item = s_item;
    if (item >= (unsigned int)num_sources) return;
    const int64_t u = __ldg(sources + item);
    int64_t* ids = idx_out + 2 * (int64_t)item * K;
    double* gd = dist_out + (int64_t)item * K;
    int reach = 0;                                      // |R(u)| - 1
    if (u >= 0 && u < num_nodes) {
      const int src = (int)u;
      // with the bitmap, the row is read only at vertices the search claims and writes: it needs no reset
      if (SMEM_VISITED)
        for (int k = threadIdx.x; k < words; k += blockDim.x) s_visited[k] = k == src / 32 ? 1u << (src & 31) : 0u;
      else
        for (int v = threadIdx.x; v < num_nodes; v += blockDim.x) row[v] = v == src ? 0 : -1;
      if (threadIdx.x == 0) {
        queue[0] = src;
        s_count[0] = 0;
        s_count[1] = 0;
        s_count[2] = 1;
      }
      __syncthreads();
      reach = hop_bfs_levels<SMEM_VISITED>(num_nodes, adj_ptr, adj_idx, row, s_visited, queue, s_count, status) - 1;
    } else if (threadIdx.x == 0 && status) {
      atomicOr(status, SYMPA_STATUS_BAD_INDEX);
    }
    if (reach == 0) {
      if (threadIdx.x == 0 && status && u >= 0 && u < num_nodes) atomicOr(status, SYMPA_STATUS_NO_PAIR);
      for (int64_t k = threadIdx.x; k < K; k += blockDim.x) {
        ids[2 * k] = u;
        ids[2 * k + 1] = u;
        gd[k] = 0.0;
      }
      continue;
    }
    const int src = (int)u;
    // bitmap of R(u) \ {u}
    if (SMEM_VISITED) {
      if (threadIdx.x == 0) s_visited[src >> 5] &= ~(1u << (src & 31));
    } else {
      for (int w = warp; w < words; w += nwarps) {
        const int v = 32 * w + lane;
        const unsigned b = __ballot_sync(full, v < num_nodes && __ldcg(row + v) > 0);
        if (lane == 0) bits[w] = b;
      }
    }
    __syncthreads();
    // exclusive popcount prefix over the words: a contiguous run of words per thread, scanned across the CTA
    const int per = (words + blockDim.x - 1) / blockDim.x;
    const int w0 = min(words, (int)threadIdx.x * per), w1 = min(words, w0 + per);
    int mine = 0;
    for (int w = w0; w < w1; ++w) mine += __popc(bits[w]);
    int incl = mine;
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(full, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) s_scan[warp] = incl;
    __syncthreads();
    int before = incl - mine;
    for (int k = 0; k < warp; ++k) before += s_scan[k];
    for (int w = w0; w < w1; ++w) {
      prefix[w] = before;
      before += __popc(bits[w]);
    }
    __syncthreads();
    for (int64_t k = threadIdx.x; k < K; k += blockDim.x) {
      const int r = (int)__umul64hi(sample_hash(seed, epoch, 0, (uint64_t)u, (uint64_t)k), (uint64_t)reach);
      int lo = 0, hi = words - 1;                       // the last word whose prefix is <= r holds draw r
      while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldcg(prefix + mid) <= r) lo = mid;
        else hi = mid - 1;
      }
      const int dst = 32 * lo + select_bit(bits[lo], r - __ldcg(prefix + lo));
      ids[2 * k] = u;
      ids[2 * k + 1] = dst;
      gd[k] = (double)__ldcg(row + dst);
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
