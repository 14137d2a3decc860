// Exact k-nearest-neighbour queries over rows of a distance matrix (sympa_dist_rows, sympa_row_topk).
//
//   query_rows_index_kernel   index pairs (queries[r], j) of a (query_count x num_rows) block, in the row-major
//                             order and with the i == j substitution of all_pairs_index_kernel, so that a query
//                             row is computed by the same pair kernels as the matrix row and is bit-identical to it
//   query_rows_fixup_kernel   one CTA per row: the zero at column queries[r], or NaN over a row whose query lies
//                             outside the table (its pairs were rejected by the pair kernels, which never read
//                             outside the table)
//   topk_select_kernel        several CTAs per row (the grid fills the GPU even for one long row): each scans its
//                             column slice once, keeping the candidates that beat a running threshold in shared
//                             memory; a full buffer is sorted, cut to k and the threshold tightened to its k-th
//                             entry; the CTA's k best go to the workspace.  The buffer (knn_buffer_entries) holds k
//                             survivors, k more candidates and one tile: with fewer than k of slack a sort would
//                             follow nearly every tile once k approaches the tile size
//   topk_merge_kernel         one CTA per row: the same selection over the splits x k candidates of the row
// The order is total: (value with -0.0 read as +0.0, column), so the k smallest are unique and do not depend on
// the split, the block or the launch shape.  NaN entries are never candidates.
// Workspace: [row_count x splits x k] {key, column} pairs of 16 bytes, column -1 for an empty slot.
#pragma once

#include <math.h>
#include <stdint.h>

namespace sympa {

// k is capped so that the largest buffer, 2 k + one tile = 3072 candidates of 16 bytes (48 KB), sorts in the shared
// memory of one CTA with room for four CTAs per SM
#define SY_KNN_MAX_K 1024
#define SY_KNN_THREADS 256
#define SY_KNN_ITEMS 4                                   // entries per thread and tile
#define SY_KNN_TILE (SY_KNN_THREADS * SY_KNN_ITEMS)
#define SY_KNN_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull           // above the key of every non-NaN double

// candidates of the shared-memory buffer for a given k (16 bytes each): at least 2 k + one tile
inline int knn_buffer_entries(int64_t k) { return 2 * (int)k + SY_KNN_TILE > 2048 ? 2 * (int)k + SY_KNN_TILE : 2048; }

// ascending unsigned order of the keys = ascending order of the (non-NaN) doubles, -0.0 equal to +0.0
__device__ __forceinline__ unsigned long long knn_key(double x) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(x == 0.0 ? 0.0 : x);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ bool knn_less(unsigned long long ka, long long ca, unsigned long long kb, long long cb) {
  return ka < kb || (ka == kb && ca < cb);
}

// ascending sort of (key, col)[0, m) by (key, col): the network of ap_bitonic_sort on 16-byte entries
__device__ inline void knn_bitonic_sort(unsigned long long* key, long long* col, int m) {
  int p2 = 1;
  while (p2 < m) p2 <<= 1;
  for (int k = 2; k <= p2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < (p2 >> 1); t += blockDim.x) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int l = (j == (k >> 1)) ? (i ^ (k - 1)) : (i | j);
        if (l < m) {
          const unsigned long long kx = key[i], ky = key[l];
          const long long cx = col[i], cy = col[l];
          if (knn_less(ky, cy, kx, cx)) {
            key[i] = ky;
            col[i] = cy;
            key[l] = kx;
            col[l] = cx;
          }
        }
      }
      __syncthreads();
    }
  }
}

// The selection shared by both kernels.  load(e, &key, &col) fetches entry e of [0, count) and returns false for
// one that is not a candidate.  On return the CTA's best min(k, candidates) entries sit sorted in s_key / s_col
// and *s_n holds their number.
// buf: the buffer's entries, >= 2 k + SY_KNN_TILE.
template <typename Load>
__device__ inline void knn_select(int64_t count, int k, int buf, Load load, unsigned long long* s_key, long long* s_col,
                                  int* s_n, unsigned long long* s_thr_key, long long* s_thr_col) {
  if (threadIdx.x == 0) {
    *s_n = 0;
    *s_thr_key = SY_KNN_EMPTY_KEY;
    *s_thr_col = INT64_MAX;
  }
  __syncthreads();
  for (int64_t t0 = 0; t0 < count; t0 += SY_KNN_TILE) {
    const unsigned long long tk = *s_thr_key;
    const long long tc = *s_thr_col;
    unsigned long long key[SY_KNN_ITEMS];
    long long col[SY_KNN_ITEMS];
    bool hit[SY_KNN_ITEMS];
    int pass = 0;
#pragma unroll
    for (int i = 0; i < SY_KNN_ITEMS; ++i) {
      const int64_t e = t0 + i * SY_KNN_THREADS + threadIdx.x;
      hit[i] = e < count && load(e, key + i, col + i) && knn_less(key[i], col[i], tk, tc);
      pass += hit[i];
    }
    if (pass) {                      // the buffer holds at most buf - SY_KNN_TILE entries here: a whole tile fits
      int at = atomicAdd(s_n, pass);
#pragma unroll
      for (int i = 0; i < SY_KNN_ITEMS; ++i)
        if (hit[i]) {
          s_key[at] = key[i];
          s_col[at] = col[i];
          ++at;
        }
    }
    __syncthreads();
    const int m = *s_n;
    __syncthreads();                 // every thread has read the count before anyone appends or rewrites it
    if (m > buf - SY_KNN_TILE) {
      knn_bitonic_sort(s_key, s_col, m);
      if (threadIdx.x == 0) {
        *s_n = k;                    // m > buf - SY_KNN_TILE >= 2 k
        *s_thr_key = s_key[k - 1];
        *s_thr_col = s_col[k - 1];
      }
      __syncthreads();
    }
  }
  const int m = *s_n;
  knn_bitonic_sort(s_key, s_col, m);
  if (threadIdx.x == 0 && m > k) *s_n = k;
  __syncthreads();
}

// grid: row_count * splits CTAs, CTA b handles row b / splits, columns of slice b % splits; dynamic shared memory:
// the buffer of buf keys, then buf columns
__global__ void __launch_bounds__(SY_KNN_THREADS) topk_select_kernel(int64_t num_cols, int splits, int k, int buf,
                                                                     const double* __restrict__ dist,
                                                                     const int64_t* __restrict__ exclude,
                                                                     longlong2* __restrict__ cand,
                                                                     unsigned int* __restrict__ status) {
  extern __shared__ unsigned long long knn_smem[];
  unsigned long long* s_key = knn_smem;
  long long* s_col = reinterpret_cast<long long*>(knn_smem + buf);
  __shared__ int s_n, s_nan;
  __shared__ unsigned long long s_thr_key;
  __shared__ long long s_thr_col;
  const int64_t r = blockIdx.x / splits;
  const int64_t part = blockIdx.x - r * splits;
  const int64_t per = (num_cols + splits - 1) / splits;
  const int64_t c0 = part * per < num_cols ? part * per : num_cols;
  const int64_t c1 = c0 + per < num_cols ? c0 + per : num_cols;
  const double* row = dist + r * num_cols + c0;
  const int64_t skip = exclude ? __ldg(exclude + r) - c0 : -1;
  if (threadIdx.x == 0) s_nan = 0;
  int nan = 0;
  knn_select(c1 - c0, k, buf,
             [&](int64_t e, unsigned long long* kk, long long* cc) {
               const double x = __ldcs(row + e);
               if (e == skip) return false;
               if (isnan(x)) {
                 nan = 1;
                 return false;
               }
               *kk = knn_key(x);
               *cc = c0 + e;
               return true;
             },
             s_key, s_col, &s_n, &s_thr_key, &s_thr_col);
  if (nan) s_nan = 1;
  __syncthreads();
  longlong2* out = cand + (int64_t)blockIdx.x * k;
  for (int i = threadIdx.x; i < k; i += blockDim.x)
    out[i] = i < s_n ? make_longlong2((long long)s_key[i], s_col[i]) : make_longlong2((long long)SY_KNN_EMPTY_KEY, -1);
  if (threadIdx.x == 0 && s_nan && status) atomicOr(status, SYMPA_STATUS_NON_FINITE);
}

// grid: row_count CTAs, shared memory as topk_select_kernel.  The distance of a selected column is read back from
// the block, so that -0.0 stays -0.0.
__global__ void __launch_bounds__(SY_KNN_THREADS) topk_merge_kernel(int64_t num_cols, int splits, int k, int buf,
                                                                    const double* __restrict__ dist,
                                                                    const longlong2* __restrict__ cand,
                                                                    int64_t* __restrict__ ids_out,
                                                                    double* __restrict__ dist_out) {
  extern __shared__ unsigned long long knn_smem[];
  unsigned long long* s_key = knn_smem;
  long long* s_col = reinterpret_cast<long long*>(knn_smem + buf);
  __shared__ int s_n;
  __shared__ unsigned long long s_thr_key;
  __shared__ long long s_thr_col;
  const int64_t r = blockIdx.x;
  const longlong2* c = cand + r * splits * (int64_t)k;
  knn_select((int64_t)splits * k, k, buf,
             [&](int64_t e, unsigned long long* kk, long long* cc) {
               const longlong2 v = c[e];
               if (v.y < 0) return false;
               *kk = (unsigned long long)v.x;
               *cc = v.y;
               return true;
             },
             s_key, s_col, &s_n, &s_thr_key, &s_thr_col);
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const bool hit = i < s_n;
    ids_out[r * k + i] = hit ? s_col[i] : -1;
    dist_out[r * k + i] = hit ? dist[r * num_cols + s_col[i]] : NAN;
  }
}

// index pairs of a block of query rows: pair t of the chunk is entry first + t of the row-major
// (query_count x num_rows) block whose row r is node queries[r], with all_pairs_index_kernel's substitution on the
// diagonal.  A query outside [0, num_rows) is passed through: the pair kernels reject it.
__global__ void __launch_bounds__(256) query_rows_index_kernel(int64_t first, int64_t count, int64_t num_rows,
                                                               const int64_t* __restrict__ queries,
                                                               longlong2* __restrict__ idx) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < count; t += stride) {
    const int64_t e = first + t;
    const int64_t r = e / num_rows;
    const int64_t j = e - r * num_rows;
    int64_t i = __ldg(queries + r);
    if (i == j) i = (i + 1) % num_rows;
    idx[t] = make_longlong2(i, j);
  }
}

__global__ void __launch_bounds__(256) query_rows_fixup_kernel(int64_t query_count, int64_t num_rows,
                                                               const int64_t* __restrict__ queries,
                                                               double* __restrict__ out, unsigned int* __restrict__ status) {
  for (int64_t r = blockIdx.x; r < query_count; r += gridDim.x) {
    const int64_t q = __ldg(queries + r);
    double* row = out + r * num_rows;
    if (q >= 0 && q < num_rows) {
      if (threadIdx.x == 0) row[q] = 0.0;
    } else {
      for (int64_t j = threadIdx.x; j < num_rows; j += blockDim.x) row[j] = NAN;
      if (threadIdx.x == 0 && status) atomicOr(status, SYMPA_STATUS_BAD_INDEX);
    }
  }
}

}  // namespace sympa
