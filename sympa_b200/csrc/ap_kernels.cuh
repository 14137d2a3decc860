// Graph-reconstruction average precision of rows of a distance matrix (sympa_average_precision).
//
//   AP(u) = 1/|N(u)| sum_{v in N(u)} |{v' in N(u) : d(u,v') <= d(u,v)}| / |{w != u : d(u,w) <= d(u,v)}|
//
// Three launches per block of rows, all counts integers so that the only floating-point sum of a row runs
// in one fixed order and a row's value does not depend on the block it came in or on the launch shape:
//   ap_prepare_kernel  one CTA per row: gathers the row's neighbour distances from the block itself, sorts
//                      them ascending into the workspace, zeroes the row's bin counters
//   ap_count_kernel    several CTAs per row (the grid fills the GPU even for a handful of long rows): every
//                      column w != u goes to the bin of its lower bound among the sorted neighbour distances,
//                      counted in shared memory and flushed to the row's 64-bit counters with integer atomics
//   ap_finish_kernel   one thread per row: rank_j = prefix sum of the bins, AP = sum_j ub_j / rank_j / m in
//                      ascending j (ub_j: neighbours at distance <= s_j, i.e. the end of s_j's tie group)
// Workspace (8-byte words): [row_count x {valid degree, flags}] [sorted distances] [bin counters], the last two
// indexed by adj_ptr[u] - adj_ptr[row_begin].
#pragma once

#include <math.h>
#include <stdint.h>

namespace sympa {

// neighbour lists up to this length are searched in shared memory by the count kernel and sorted there by
// the prepare kernel; longer ones (hubs) are sorted and searched in the workspace
#define SY_AP_SMEM_CAP 2048
#define SY_AP_THREADS 256
#define SY_AP_FLAG_NAN 1ull

// Ascending sort of a[0, m) by the all-ascending ("flip") form of the bitonic network: the elements past m act
// as +inf padding up to the next power of two, and every compare-exchange whose upper partner lies past m is a
// no-op, so it is skipped.  Called by the whole CTA; `a` is shared or global memory of this CTA only.
__device__ inline void ap_bitonic_sort(double* a, int64_t m) {
  int64_t p2 = 1;
  while (p2 < m) p2 <<= 1;
  for (int64_t k = 2; k <= p2; k <<= 1) {
    for (int64_t j = k >> 1; j > 0; j >>= 1) {
      for (int64_t t = threadIdx.x; t < (p2 >> 1); t += blockDim.x) {
        // t-th index with bit j clear, and its partner: i ^ (k - 1) for the flip step, i ^ j afterwards
        const int64_t i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int64_t l = (j == (k >> 1)) ? (i ^ (k - 1)) : (i | j);
        if (l < m) {
          const double x = a[i], y = a[l];
          if (y < x) {
            a[i] = y;
            a[l] = x;
          }
        }
      }
      __syncthreads();
    }
  }
}

__global__ void __launch_bounds__(SY_AP_THREADS) ap_prepare_kernel(int64_t row_begin, int64_t num_cols,
                                                                   const double* __restrict__ dist,
                                                                   const int64_t* __restrict__ adj_ptr,
                                                                   const int64_t* __restrict__ adj_idx, int64_t cap,
                                                                   int64_t* __restrict__ meta, double* __restrict__ sorted,
                                                                   unsigned long long* __restrict__ counts,
                                                                   unsigned int* __restrict__ status) {
  __shared__ double s_val[SY_AP_SMEM_CAP];
  __shared__ int s_invalid;
  __shared__ int s_nan;
  const int64_t r = blockIdx.x;
  const int64_t u = row_begin + r;
  const int64_t base = __ldg(adj_ptr + row_begin);
  const int64_t p0 = __ldg(adj_ptr + u), p1 = __ldg(adj_ptr + u + 1);
  if (p0 < base || p1 < p0 || p1 - base > cap) {   // malformed row pointer: the row has no usable neighbour
    if (threadIdx.x == 0) {
      meta[2 * r] = 0;
      meta[2 * r + 1] = 0;
      if (status) atomicOr(status, SYMPA_STATUS_BAD_INDEX);
    }
    return;
  }
  const int64_t m = p1 - p0;
  if (threadIdx.x == 0) {
    s_invalid = 0;
    s_nan = 0;
  }
  __syncthreads();
  const bool in_smem = m <= SY_AP_SMEM_CAP;
  double* out = sorted + (p0 - base);
  double* a = in_smem ? s_val : out;
  const double* row = dist + r * num_cols;
  int invalid = 0, nan = 0;
  for (int64_t j = threadIdx.x; j < m; j += blockDim.x) {
    const int64_t v = __ldg(adj_idx + p0 + j);
    double x = INFINITY;            // excluded entries sort to the end and are cut off by the valid degree
    if (v < 0 || v >= num_cols) {
      ++invalid;
      if (status) atomicOr(status, SYMPA_STATUS_BAD_INDEX);
    } else if (v == u) {
      ++invalid;
    } else {
      x = __ldg(row + v);
      if (isnan(x)) {
        nan = 1;
        x = INFINITY;
      }
    }
    a[j] = x;
    counts[p0 - base + j] = 0ull;
  }
  if (invalid) atomicAdd(&s_invalid, invalid);
  if (nan) s_nan = 1;
  __syncthreads();
  ap_bitonic_sort(a, m);
  if (in_smem)
    for (int64_t j = threadIdx.x; j < m; j += blockDim.x) out[j] = a[j];
  if (threadIdx.x == 0) {
    meta[2 * r] = m - s_invalid;
    meta[2 * r + 1] = s_nan ? (int64_t)SY_AP_FLAG_NAN : 0;
    if (s_nan && status) atomicOr(status, SYMPA_STATUS_NON_FINITE);
  }
}

// first index j in [0, m) with s[j] >= x (m when there is none)
__device__ __forceinline__ int64_t ap_lower_bound(const double* s, int64_t m, double x) {
  int64_t lo = 0, hi = m;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (s[mid] < x)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

// grid: row_count * splits CTAs, CTA b handles row b / splits, columns of slice b % splits
__global__ void __launch_bounds__(SY_AP_THREADS) ap_count_kernel(int64_t row_begin, int64_t num_cols, int splits,
                                                                 const double* __restrict__ dist,
                                                                 const int64_t* __restrict__ adj_ptr,
                                                                 int64_t* __restrict__ meta, const double* __restrict__ sorted,
                                                                 unsigned long long* __restrict__ counts,
                                                                 unsigned int* __restrict__ status) {
  __shared__ double s_val[SY_AP_SMEM_CAP];
  __shared__ unsigned long long s_cnt[SY_AP_SMEM_CAP];
  __shared__ int s_nan;
  const int64_t r = blockIdx.x / splits;
  const int64_t part = blockIdx.x - r * splits;
  const int64_t m = meta[2 * r];
  if (m <= 0) return;
  const int64_t u = row_begin + r;
  const int64_t off = __ldg(adj_ptr + u) - __ldg(adj_ptr + row_begin);
  const double* s = sorted + off;
  unsigned long long* cnt = counts + off;
  const bool in_smem = m <= SY_AP_SMEM_CAP;
  if (in_smem) {
    for (int64_t j = threadIdx.x; j < m; j += blockDim.x) {
      s_val[j] = s[j];
      s_cnt[j] = 0ull;
    }
    s = s_val;
  }
  if (threadIdx.x == 0) s_nan = 0;
  __syncthreads();
  unsigned long long* c = in_smem ? s_cnt : cnt;
  const int64_t per = (num_cols + splits - 1) / splits;
  const int64_t c0 = part * per;
  const int64_t c1 = c0 + per < num_cols ? c0 + per : num_cols;
  const double* row = dist + r * num_cols;
  // runs of equal bins are counted in a register first: with few neighbours most columns share a bin
  int64_t run_bin = -1;
  unsigned long long run = 0;
  int nan = 0;
  for (int64_t w = c0 + threadIdx.x; w < c1; w += blockDim.x) {
    const double x = __ldcs(row + w);
    if (w == u) continue;
    if (isnan(x)) {
      nan = 1;
      continue;
    }
    const int64_t b = ap_lower_bound(s, m, x);
    if (b >= m) continue;           // farther than every neighbour: ranks none of them
    if (b != run_bin) {
      if (run) atomicAdd(c + run_bin, run);
      run_bin = b;
      run = 0;
    }
    ++run;
  }
  if (run) atomicAdd(c + run_bin, run);
  if (nan) s_nan = 1;
  __syncthreads();
  if (in_smem)
    for (int64_t j = threadIdx.x; j < m; j += blockDim.x)
      if (s_cnt[j]) atomicAdd(cnt + j, s_cnt[j]);
  if (threadIdx.x == 0 && s_nan) {
    atomicOr(reinterpret_cast<unsigned long long*>(meta + 2 * r + 1), SY_AP_FLAG_NAN);
    if (status) atomicOr(status, SYMPA_STATUS_NON_FINITE);
  }
}

__global__ void __launch_bounds__(SY_AP_THREADS) ap_finish_kernel(int64_t row_begin, int64_t row_count,
                                                                  const int64_t* __restrict__ adj_ptr,
                                                                  const int64_t* __restrict__ meta,
                                                                  const double* __restrict__ sorted,
                                                                  const unsigned long long* __restrict__ counts,
                                                                  double* __restrict__ ap_out) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= row_count) return;
  const int64_t m = meta[2 * r];
  if (m <= 0 || (meta[2 * r + 1] & (int64_t)SY_AP_FLAG_NAN)) {
    ap_out[r] = NAN;
    return;
  }
  const int64_t off = __ldg(adj_ptr + row_begin + r) - __ldg(adj_ptr + row_begin);
  const double* s = sorted + off;
  const unsigned long long* cnt = counts + off;
  double sum = 0.0;
  unsigned long long rank = 0;
  for (int64_t a = 0; a < m;) {
    int64_t e = a + 1;              // [a, e): one tie group
    while (e < m && s[e] == s[a]) ++e;
    for (int64_t j = a; j < e; ++j) {
      rank += cnt[j];
      sum += (double)e / (double)rank;
    }
    a = e;
  }
  ap_out[r] = sum / (double)m;
}

}  // namespace sympa
