// Filtered ranks of held-out targets among all nodes (sympa_target_ranks), for link-prediction evaluation.
//
// For block row r with query u = queries[r], target v, filter row F(u) and competitors
// C = {w : w != u, w != v, w not in F(u)}:
//   lt = |{w in C : d(u,w) < d(u,v)}|,   le = |{w in C : d(u,w) <= d(u,v)}|
// Three launches per block, all counts integers, so a pair's result does not depend on the block, offset or launch
// shape:
//   rank_prepare_kernel  one CTA per row: gathers the distances of the row's targets, sorts them ascending into the
//                        workspace (ap_bitonic_sort), zeroes the row's two bin arrays
//   rank_count_kernel    several CTAs per row: every column w != u goes to the bin b of its lower bound among the
//                        sorted target distances s; le_bins[b] counts it, eq_bins[b] too when s[b] == d(u,w).  The
//                        row is read once, as in ap_count_kernel, counting in shared memory with integer atomics
//   rank_finish_kernel   one CTA per row: takes the columns of F(u) back out of the bins, turns le_bins into its
//                        prefix sum, then for target v at lower bound a: le = le_bins[a] and lt = le - eq_bins[a]
//                        (the columns at exactly d(u,v)), minus v itself from le when v is not in F(u)
// Every column of one tie group of s lands on the group's first index, so any target of the group reads the same
// bins.  A NaN in the row (w != u) flags the row: its pairs get lt = le = -1.
// Workspace (8-byte words): [row_count flags] [sorted distances] [le bins] [eq bins], the last three indexed by
// target_ptr[r] - target_ptr[0].
#pragma once

#include <math.h>
#include <stdint.h>

#include "ap_kernels.cuh"

namespace sympa {

// targets of a row up to this number are searched and counted in shared memory by the count kernel; longer rows
// count in the workspace
#define SY_RANK_SMEM_CAP 2048
#define SY_RANK_THREADS 256
#define SY_RANK_FLAG_NAN 1ull
#define SY_RANK_FLAG_SKIP 2ull       // the row is not evaluated: a query outside [0, num_cols) or no workspace room

__global__ void __launch_bounds__(SY_RANK_THREADS) rank_prepare_kernel(int64_t num_cols, const double* __restrict__ dist,
                                                                       const int64_t* __restrict__ queries,
                                                                       const int64_t* __restrict__ target_ptr,
                                                                       const int64_t* __restrict__ target_idx, int64_t cap,
                                                                       unsigned long long* __restrict__ flags,
                                                                       double* __restrict__ sorted,
                                                                       unsigned long long* __restrict__ le_bins,
                                                                       unsigned long long* __restrict__ eq_bins,
                                                                       unsigned int* __restrict__ status) {
  __shared__ double s_val[SY_RANK_SMEM_CAP];
  const int64_t r = blockIdx.x;
  const int64_t u = __ldg(queries + r);
  const int64_t base = __ldg(target_ptr);
  const int64_t p0 = __ldg(target_ptr + r), p1 = __ldg(target_ptr + r + 1);
  if (u < 0 || u >= num_cols || p0 < base || p1 < p0 || p1 - base > cap) {
    if (threadIdx.x == 0) {
      flags[r] = SY_RANK_FLAG_SKIP;
      if (status) atomicOr(status, SYMPA_STATUS_BAD_INDEX);
    }
    return;
  }
  if (threadIdx.x == 0) flags[r] = 0;
  const int64_t m = p1 - p0;
  const bool in_smem = m <= SY_RANK_SMEM_CAP;
  double* out = sorted + (p0 - base);
  double* a = in_smem ? s_val : out;
  const double* row = dist + r * num_cols;
  for (int64_t j = threadIdx.x; j < m; j += blockDim.x) {
    const int64_t v = __ldg(target_idx + p0 + j);
    double x = INFINITY;              // a bad target sorts last; its own result is -1 (rank_finish_kernel)
    if (v < 0 || v >= num_cols) {
      if (status) atomicOr(status, SYMPA_STATUS_BAD_INDEX);
    } else {
      x = __ldg(row + v);
      if (isnan(x)) x = INFINITY;     // the count kernel flags the row
    }
    a[j] = x;
    le_bins[p0 - base + j] = 0ull;
    eq_bins[p0 - base + j] = 0ull;
  }
  __syncthreads();
  ap_bitonic_sort(a, m);
  if (in_smem)
    for (int64_t j = threadIdx.x; j < m; j += blockDim.x) out[j] = a[j];
}

// one run of equal bins, counted in registers, flushed to the bins c_le / c_eq (shared 32-bit or global 64-bit)
template <typename C>
__device__ __forceinline__ void rank_flush(C* c_le, C* c_eq, int64_t bin, unsigned long long le, unsigned long long eq) {
  if (le) atomicAdd(c_le + bin, (C)le);
  if (eq) atomicAdd(c_eq + bin, (C)eq);
}

// grid: row_count * splits CTAs, CTA b handles row b / splits, columns of slice b % splits (at most 2^32 - 1 columns,
// so that the shared 32-bit bins cannot overflow)
__global__ void __launch_bounds__(SY_RANK_THREADS) rank_count_kernel(int64_t num_cols, int splits,
                                                                     const double* __restrict__ dist,
                                                                     const int64_t* __restrict__ queries,
                                                                     const int64_t* __restrict__ target_ptr,
                                                                     unsigned long long* __restrict__ flags,
                                                                     const double* __restrict__ sorted,
                                                                     unsigned long long* __restrict__ le_bins,
                                                                     unsigned long long* __restrict__ eq_bins,
                                                                     unsigned int* __restrict__ status) {
  __shared__ double s_val[SY_RANK_SMEM_CAP];
  __shared__ unsigned int s_le[SY_RANK_SMEM_CAP];
  __shared__ unsigned int s_eq[SY_RANK_SMEM_CAP];
  __shared__ int s_nan;
  const int64_t r = blockIdx.x / splits;
  const int64_t part = blockIdx.x - r * splits;
  if (flags[r] & SY_RANK_FLAG_SKIP) return;
  const int64_t base = __ldg(target_ptr);
  const int64_t p0 = __ldg(target_ptr + r);
  const int64_t m = __ldg(target_ptr + r + 1) - p0;
  if (m <= 0) return;                 // no targets: the row is not read
  const int64_t u = __ldg(queries + r);
  const double* s = sorted + (p0 - base);
  const bool in_smem = m <= SY_RANK_SMEM_CAP;
  if (in_smem) {
    for (int64_t j = threadIdx.x; j < m; j += blockDim.x) {
      s_val[j] = s[j];
      s_le[j] = 0u;
      s_eq[j] = 0u;
    }
    s = s_val;
  }
  if (threadIdx.x == 0) s_nan = 0;
  __syncthreads();
  unsigned long long* g_le = le_bins + (p0 - base);
  unsigned long long* g_eq = eq_bins + (p0 - base);
  const int64_t per = (num_cols + splits - 1) / splits;
  const int64_t c0 = part * per;
  const int64_t c1 = c0 + per < num_cols ? c0 + per : num_cols;
  const double* row = dist + r * num_cols;
  // with few targets most columns share a bin: runs of equal bins are counted in registers first
  int64_t run_bin = -1;
  unsigned long long run_le = 0, run_eq = 0;
  int nan = 0;
  for (int64_t w = c0 + threadIdx.x; w < c1; w += blockDim.x) {
    const double x = __ldcs(row + w);
    if (w == u) continue;
    if (isnan(x)) {
      nan = 1;
      continue;
    }
    const int64_t b = ap_lower_bound(s, m, x);
    if (b >= m) continue;             // farther than every target: counts for none of them
    if (b != run_bin) {
      if (in_smem)
        rank_flush(s_le, s_eq, run_bin, run_le, run_eq);
      else
        rank_flush(g_le, g_eq, run_bin, run_le, run_eq);
      run_bin = b;
      run_le = run_eq = 0;
    }
    ++run_le;
    run_eq += s[b] == x;
  }
  if (in_smem)
    rank_flush(s_le, s_eq, run_bin, run_le, run_eq);
  else
    rank_flush(g_le, g_eq, run_bin, run_le, run_eq);
  if (nan) s_nan = 1;
  __syncthreads();
  if (in_smem)
    for (int64_t j = threadIdx.x; j < m; j += blockDim.x) {
      if (s_le[j]) atomicAdd(g_le + j, (unsigned long long)s_le[j]);
      if (s_eq[j]) atomicAdd(g_eq + j, (unsigned long long)s_eq[j]);
    }
  if (threadIdx.x == 0 && s_nan) {
    atomicOr(flags + r, SY_RANK_FLAG_NAN);
    if (status) atomicOr(status, SYMPA_STATUS_NON_FINITE);
  }
}

// in-place inclusive prefix sum of a[0, m), called by the whole CTA (blockDim.x a multiple of 32, at most 1024)
__device__ inline void rank_inclusive_scan(unsigned long long* a, int64_t m) {
  __shared__ unsigned long long s_warp[32];
  __shared__ unsigned long long s_carry;
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = 0ull;
  __syncthreads();
  for (int64_t c0 = 0; c0 < m; c0 += blockDim.x) {
    const int64_t i = c0 + threadIdx.x;
    unsigned long long v = i < m ? a[i] : 0ull;
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long y = __shfl_up_sync(full, v, o);
      if (lane >= o) v += y;
    }
    if (lane == 31) s_warp[warp] = v;
    __syncthreads();
    unsigned long long before = s_carry;
    for (int k = 0; k < warp; ++k) before += s_warp[k];
    if (i < m) a[i] = before + v;
    __syncthreads();                  // every thread has read s_carry and s_warp
    if (threadIdx.x == blockDim.x - 1) s_carry = before + v;
    __syncthreads();
  }
}

// first index j in [0, m) with s[j] >= x, for a sorted int64 array
__device__ __forceinline__ int64_t rank_lower_bound_i64(const int64_t* s, int64_t m, int64_t x) {
  int64_t lo = 0, hi = m;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(s + mid) < x)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo;
}

// grid: row_count CTAs
__global__ void __launch_bounds__(SY_RANK_THREADS) rank_finish_kernel(int64_t num_cols, const double* __restrict__ dist,
                                                                      const int64_t* __restrict__ queries,
                                                                      const int64_t* __restrict__ target_ptr,
                                                                      const int64_t* __restrict__ target_idx,
                                                                      const int64_t* __restrict__ filter_ptr,
                                                                      const int64_t* __restrict__ filter_idx,
                                                                      const unsigned long long* __restrict__ flags,
                                                                      const double* __restrict__ sorted,
                                                                      unsigned long long* __restrict__ le_bins,
                                                                      unsigned long long* __restrict__ eq_bins,
                                                                      int64_t* __restrict__ lt_out, int64_t* __restrict__ le_out,
                                                                      unsigned int* __restrict__ status) {
  const int64_t r = blockIdx.x;
  const int64_t base = __ldg(target_ptr);
  const int64_t p0 = __ldg(target_ptr + r), p1 = __ldg(target_ptr + r + 1);
  if (p0 < base || p1 < p0) return;   // malformed pointers: nothing of this row can be written
  const int64_t m = p1 - p0;
  if (m == 0) return;
  if (flags[r]) {                     // NaN in the row, or not evaluated
    for (int64_t j = threadIdx.x; j < m; j += blockDim.x) {
      lt_out[p0 + j] = -1;
      le_out[p0 + j] = -1;
    }
    return;
  }
  const int64_t u = __ldg(queries + r);
  const double* s = sorted + (p0 - base);
  unsigned long long* le = le_bins + (p0 - base);
  unsigned long long* eq = eq_bins + (p0 - base);
  const double* row = dist + r * num_cols;
  const int64_t f0 = __ldg(filter_ptr + u), f1 = __ldg(filter_ptr + u + 1);
  // the filtered columns were counted like any other: take them back out
  for (int64_t i = f0 + threadIdx.x; i < f1; i += blockDim.x) {
    const int64_t w = __ldg(filter_idx + i);
    if (w < 0 || w >= num_cols) {
      if (status) atomicOr(status, SYMPA_STATUS_BAD_INDEX);
      continue;
    }
    if (w == u) continue;
    const double x = __ldg(row + w);
    const int64_t b = ap_lower_bound(s, m, x);
    if (b >= m) continue;
    atomicAdd(le + b, ~0ull);         // - 1 modulo 2^64
    if (s[b] == x) atomicAdd(eq + b, ~0ull);
  }
  __syncthreads();
  rank_inclusive_scan(le, m);
  for (int64_t j = threadIdx.x; j < m; j += blockDim.x) {
    const int64_t v = __ldg(target_idx + p0 + j);
    if (v < 0 || v >= num_cols) {
      lt_out[p0 + j] = -1;
      le_out[p0 + j] = -1;
      continue;
    }
    const double x = __ldg(row + v);
    const int64_t a = ap_lower_bound(s, m, x);
    const int64_t n_le = (int64_t)le[a];
    const int64_t n_eq = (int64_t)eq[a];
    // v itself is one of the columns at d(u,v) unless it is u or was filtered
    const int64_t k = rank_lower_bound_i64(filter_idx + f0, f1 - f0, v);
    const bool counted = v != u && !(k < f1 - f0 && __ldg(filter_idx + f0 + k) == v);
    lt_out[p0 + j] = n_le - n_eq;
    le_out[p0 + j] = n_le - (counted ? 1 : 0);
  }
}

}  // namespace sympa
