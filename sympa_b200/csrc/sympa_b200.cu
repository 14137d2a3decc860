// sympa_b200 - the C ABI declared in include/sympa_b200.h plus the element-wise backward kernels.
//
//   pair_kernel<N, KIND, MODE>   (pair_kernels.cuh)  gather -> dist (-> unit gradients | -> loss + scatter-add)
//   scale_kernel                 grad_z = grad_dist[p] * unit gradient           (materialised backward)
//   scatter_kernel               grad_table[idx] += grad_dist[p] * unit gradient (gather backward,
//                                replaces the dense index_put of sympa/embeddings.py:34's backward)
//   wsum_grad_kernel             dL/dw of the learnable wsum metric (sympa/manifolds/metrics.py:103-121)
//   ap_*_kernel                  average precision of distance-matrix rows (ap_kernels.cuh)
//   hop_bfs_kernel               graph hop distances of a block of source rows (hop_kernels.cuh)
//   sample_pairs_kernel          training pairs and their hop distances sampled per source (hop_kernels.cuh)
//   distortion_rows_kernel       graph-reconstruction distortion of distance-matrix rows (hop_kernels.cuh)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/sympa_b200.h"
#include "pair_kernels.cuh"
#include "ap_kernels.cuh"
#include "hop_kernels.cuh"

namespace sympa {

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// grad_z[p, :] = grad_dist[p] * unit[p, :]   (two operands in one launch)
__global__ void __launch_bounds__(256) scale_kernel(int64_t total2, int per2, const double* __restrict__ gd,
                                                    const double2* __restrict__ u1, const double2* __restrict__ u2,
                                                    double2* __restrict__ o1, double2* __restrict__ o2) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total2; e += stride) {
    const double g = __ldg(gd + e / per2);
    double2 a = __ldg(u1 + e), b = __ldg(u2 + e);
    o1[e] = make_double2(g * a.x, g * a.y);
    o2[e] = make_double2(g * b.x, g * b.y);
  }
}

__global__ void __launch_bounds__(256) scale_kernel1(int64_t total, int per, const double* __restrict__ gd,
                                                     const double* __restrict__ u1, const double* __restrict__ u2,
                                                     double* __restrict__ o1, double* __restrict__ o2) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
    const double g = __ldg(gd + e / per);
    o1[e] = g * __ldg(u1 + e);
    o2[e] = g * __ldg(u2 + e);
  }
}

// grad_table[idx[p, s], :] += grad_dist[p] * unit_s[p, :]
__global__ void __launch_bounds__(256) scatter_kernel(int64_t total, int per, int64_t num_rows,
                                                      const double* __restrict__ gd, const int64_t* __restrict__ idx,
                                                      const double* __restrict__ u1, const double* __restrict__ u2,
                                                      double* __restrict__ grad_table) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
    const int64_t p = e / per;
    const int c = (int)(e - p * per);
    const double g = __ldg(gd + p);
    const int64_t i1 = __ldg(idx + 2 * p), i2 = __ldg(idx + 2 * p + 1);
    if (i1 < 0 || i1 >= num_rows || i2 < 0 || i2 >= num_rows) continue;
    // (streaming loads - ld.global.cs - of the saved state measured 9 % slower here: 1.80 -> 1.97 ms)
    atomicAdd(grad_table + i1 * per + c, g * __ldg(u1 + e));
    atomicAdd(grad_table + i2 * per + c, g * __ldg(u2 + e));
  }
}

// The same two kernels for the PACKED saved state of the register kernels (state_is_packed): a point's
// unit gradient is stored as the lower triangles of its symmetric blocks; element c of the full point
// reads packed entry lut[c] (built once per block in shared memory).
__device__ __forceinline__ void build_state_lut(short* lut, int per, int n) {
  const int nn = n * n, tri_n = n * (n + 1) / 2;
  for (int c = threadIdx.x; c < per; c += blockDim.x) {
    const int m = c / nn, ij = c - m * nn, i = ij / n, j = ij - i * n;
    lut[c] = (short)(m * tri_n + (i >= j ? i * (i + 1) / 2 + j : j * (j + 1) / 2 + i));
  }
  __syncthreads();
}

__global__ void __launch_bounds__(256) scale_kernel_packed(int64_t total, int per, int per_s, int n,
                                                           const double* __restrict__ gd, const double* __restrict__ u1,
                                                           const double* __restrict__ u2, double* __restrict__ o1,
                                                           double* __restrict__ o2) {
  __shared__ short lut[2 * SYMPA_MAX_N * SYMPA_MAX_N];
  build_state_lut(lut, per, n);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
    const int64_t p = e / per;
    const int c = (int)(e - p * per);
    const double g = __ldg(gd + p);
    const int64_t off = p * per_s + lut[c];
    o1[e] = g * __ldg(u1 + off);
    o2[e] = g * __ldg(u2 + off);
  }
}

__global__ void __launch_bounds__(256) scatter_kernel_packed(int64_t total, int per, int per_s, int n, int64_t num_rows,
                                                             const double* __restrict__ gd, const int64_t* __restrict__ idx,
                                                             const double* __restrict__ u1, const double* __restrict__ u2,
                                                             double* __restrict__ grad_table) {
  __shared__ short lut[2 * SYMPA_MAX_N * SYMPA_MAX_N];
  build_state_lut(lut, per, n);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
    const int64_t p = e / per;
    const int c = (int)(e - p * per);
    const double g = __ldg(gd + p);
    const int64_t i1 = __ldg(idx + 2 * p), i2 = __ldg(idx + 2 * p + 1);
    if (i1 < 0 || i1 >= num_rows || i2 < 0 || i2 >= num_rows) continue;
    const int64_t off = p * per_s + lut[c];
    atomicAdd(grad_table + i1 * per + c, g * __ldg(u1 + off));
    atomicAdd(grad_table + i2 * per + c, g * __ldg(u2 + off));
  }
}

// Packed table gradient (sympa_dist_backward_table with a workspace): the scatter-add goes into a
// (num_rows, per_s) table of packed lower triangles - 62 % of the bytes of the dense gradient at n = 4,
// so fewer and smaller DRAM read-modify-writes and a better L2 hit rate for the random rows - with fully
// coalesced reads of the packed saved state; expand_table_kernel then writes (or adds) the dense
// symmetric rows once.
// Destination rows [row_lo, row_hi) only: the host runs the kernel in PASSES over row ranges small enough for
// the range's packed gradient rows to stay resident in L2 (the whole 168 MB table of 2^20 rows at n = 4 does
// not fit, and round 1 measured 852 B of DRAM traffic per pair - read-modify-writes of rows that had been
// evicted - against 340 B when the accumulation happens in L2 and every row is written back once).  A pass
// reads the saved state of an operand only when its row is in range, so the state is still read once overall;
// the 24 bytes of indices + upstream gradient per pair are re-read by every pass.
__global__ void __launch_bounds__(256) scatter_packed_table_kernel(int64_t total, int per_s, int64_t num_rows,
                                                                   int64_t row_lo, int64_t row_hi,
                                                                   const double* __restrict__ gd,
                                                                   const int64_t* __restrict__ idx,
                                                                   const double* __restrict__ u1,
                                                                   const double* __restrict__ u2, double* __restrict__ ws) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
    const int64_t p = e / per_s;
    const int c = (int)(e - p * per_s);
    const int64_t i1 = __ldg(idx + 2 * p), i2 = __ldg(idx + 2 * p + 1);
    if (i1 < 0 || i1 >= num_rows || i2 < 0 || i2 >= num_rows) continue;
    const bool in1 = i1 >= row_lo && i1 < row_hi, in2 = i2 >= row_lo && i2 < row_hi;
    if (!in1 && !in2) continue;
    const double g = __ldg(gd + p);
    if (in1) atomicAdd(ws + i1 * per_s + c, g * __ldg(u1 + e));
    if (in2) atomicAdd(ws + i2 * per_s + c, g * __ldg(u2 + e));
  }
}

// The same scatter over ALL destination rows (the default: one pass), written for memory-level parallelism: ncu
// showed the ranged kernel above latency-bound at full occupancy (long_scoreboard 44 per issue, DRAM at 60 % of
// its peak) - every work item was one dependent chain index -> range test -> state loads -> atomics.  Here the
// state of both operands does not wait for the indices, and U work items per thread are loaded before the first
// atomic is issued.  T is the work-item counter type (32-bit when total < 2^31: the division by per_s is a
// fifth of the 64-bit one).
template <int U, typename T>
__global__ void __launch_bounds__(256) scatter_packed_all_kernel(T total, int per_s, int64_t num_rows,
                                                                 const double* __restrict__ gd,
                                                                 const int64_t* __restrict__ idx,
                                                                 const double* __restrict__ u1,
                                                                 const double* __restrict__ u2, double* __restrict__ ws) {
  const T stride = (T)gridDim.x * (T)blockDim.x;
  const T first = (T)blockIdx.x * (T)blockDim.x + (T)threadIdx.x;
  // the stride of 64-bit counters cannot overflow; 32-bit ones are only used when total + U * stride < 2^32
  for (T e0 = first; e0 < total; e0 += (T)U * stride) {
    double a1[U], a2[U], g[U];
    int64_t i1[U], i2[U];
    int c[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const T e = e0 + (T)k * stride;
      const bool live = e < total;
      const T ee = live ? e : first;     // (in range: first < total here)
      const T p = ee / (T)per_s;
      c[k] = (int)(ee - p * (T)per_s);
      a1[k] = __ldg(u1 + ee);
      a2[k] = __ldg(u2 + ee);
      g[k] = __ldg(gd + p);
      i1[k] = __ldg(idx + 2 * (int64_t)p);
      i2[k] = __ldg(idx + 2 * (int64_t)p + 1);
      if (!live) i1[k] = -1;
    }
#pragma unroll
    for (int k = 0; k < U; ++k) {
      if (i1[k] < 0 || i1[k] >= num_rows || i2[k] < 0 || i2[k] >= num_rows) continue;
      atomicAdd(ws + i1[k] * per_s + c[k], g[k] * a1[k]);
      atomicAdd(ws + i2[k] * per_s + c[k], g[k] * a2[k]);
    }
  }
}

#ifndef SY_SCATTER_UNROLL
#define SY_SCATTER_UNROLL 4
#endif

// The same scatter confined to the SMs with %smid < sm_limit, for a caller that runs it on a side stream NEXT TO
// the forward kernel of the following chunk (ops.TableGradAccumulator): the scatter is bound by L2 atomics and
// DRAM read-modify-writes and leaves the FP64 pipes idle, the pair kernels are the opposite - but the two cannot
// share an SM (two 128-thread pair CTAs own the whole register file), so the overlap is by SM partition.  The grid
// is one full wave (8 CTAs of 256 threads per SM); CTAs that find themselves on another SM leave at once - freeing
// it for the pair kernel - and the others pull chunks of work items from a ticket counter.  Wherever the CTAs
// land the result is complete: the last CTA to leave drains the tickets that nobody took (in the worst case, no
// CTA on a chosen SM, it does all the work alone - slow, never wrong).  tickets[0] = next chunk, tickets[1] = CTAs
// that have left; both zeroed by the launcher on the same stream.
// Work items are walked without divisions: a ticket is 256 PAIRS (256 * per_s items, contiguous in the saved
// state); thread t takes the items t, t + 256, ... of the chunk, so its (pair, element) position advances by the
// constant (256 / per_s, 256 % per_s) - the partition is bound by instruction issue per SM (one item per clock and SM
// with the generic indexing of the kernels above), and every instruction saved is SM time given back to the pair kernel.
template <int U>
__global__ void __launch_bounds__(256) scatter_packed_part_kernel(int64_t num_pairs, int per_s, int64_t num_rows, int sm_limit,
                                                                  unsigned int* __restrict__ tickets,
                                                                  const double* __restrict__ gd,
                                                                  const int64_t* __restrict__ idx,
                                                                  const double* __restrict__ u1,
                                                                  const double* __restrict__ u2, double* __restrict__ ws) {
  __shared__ unsigned int s_ticket;
  __shared__ int s_last;
  unsigned int smid;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
  bool work = (int)smid < sm_limit, drain = false;
  const int t = threadIdx.x;
  const int p_first = t / per_s, c_first = t - p_first * per_s;
  const int step_p = 256 / per_s, step_c = 256 - step_p * per_s;
  const longlong2* __restrict__ idx2 = reinterpret_cast<const longlong2*>(idx);
  for (;;) {
    if (work) {
      for (;;) {
        if (t == 0) s_ticket = atomicAdd(tickets, 1u);
        __syncthreads();
        const int64_t pair0 = (int64_t)s_ticket * 256;
        __syncthreads();
        if (pair0 >= num_pairs) break;
        const int left = (num_pairs - pair0) < 256 ? (int)(num_pairs - pair0) : 256;   // pairs of this chunk
        const double* __restrict__ v1 = u1 + pair0 * per_s + t;
        const double* __restrict__ v2 = u2 + pair0 * per_s + t;
        int pl = p_first, c = c_first;
#pragma unroll 1
        for (int i0 = 0; i0 < per_s; i0 += U) {
          double a1[U], a2[U], g[U];
          longlong2 ij[U];
          int cc[U];
#pragma unroll
          for (int k = 0; k < U; ++k) {
            const bool live = i0 + k < per_s && pl < left;
            // (an item past the end of a ragged last chunk reads element 0 of the state instead: always mapped)
            const int64_t pp = pair0 + (live ? pl : 0);
            a1[k] = __ldg(live ? v1 + (i0 + k) * 256 : u1);
            a2[k] = __ldg(live ? v2 + (i0 + k) * 256 : u2);
            g[k] = __ldg(gd + pp);
            ij[k] = __ldg(idx2 + pp);
            if (!live) ij[k].x = -1;
            cc[k] = c;
            pl += step_p;
            c += step_c;
            if (c >= per_s) {
              c -= per_s;
              ++pl;
            }
          }
#pragma unroll
          for (int k = 0; k < U; ++k) {
            if (ij[k].x < 0 || ij[k].x >= num_rows || ij[k].y < 0 || ij[k].y >= num_rows) continue;
            atomicAdd(ws + ij[k].x * per_s + cc[k], g[k] * a1[k]);
            atomicAdd(ws + ij[k].y * per_s + cc[k], g[k] * a2[k]);
          }
        }
      }
    }
    if (drain) return;
    // leaving: the last CTA of the grid to get here checks that every ticket was taken
    if (t == 0) s_last = (atomicAdd(tickets + 1, 1u) == gridDim.x - 1) ? 1 : 0;
    __syncthreads();
    if (!s_last || work) return;   // a working CTA only leaves when the tickets are exhausted: nothing to drain
    work = drain = true;           // the last CTA sat on an SM outside the partition: drain (normally nothing is left)
  }
}

__global__ void __launch_bounds__(256) expand_table_kernel(int64_t total, int per, int per_s, int n, int overwrite,
                                                           const double* __restrict__ ws, double* __restrict__ grad_table) {
  __shared__ short lut[2 * SYMPA_MAX_N * SYMPA_MAX_N];
  build_state_lut(lut, per, n);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  if (per % 2 == 0) {  // two consecutive elements of a row per thread: 16-byte stores
    double2* gt2 = reinterpret_cast<double2*>(grad_table);
    const int per2 = per / 2;
    for (int64_t e2 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e2 < total / 2; e2 += stride) {
      const int64_t r = e2 / per2;
      const int c = 2 * (int)(e2 - r * per2);
      const double* row = ws + r * per_s;
      double2 v = make_double2(__ldg(row + lut[c]), __ldg(row + lut[c + 1]));
      if (!overwrite) {
        const double2 o = gt2[e2];
        v.x += o.x;
        v.y += o.y;
      }
      gt2[e2] = v;
    }
    return;
  }
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
    const int64_t r = e / per;
    const int c = (int)(e - r * per);
    const double v = __ldg(ws + r * per_s + lut[c]);
    grad_table[e] = overwrite ? v : grad_table[e] + v;
  }
}

// grad_w[k] += sum_p grad_dist[p] * vvd[p, k] * (w_k > 0)      (relu backward, metrics.py:118)
__global__ void __launch_bounds__(256) wsum_grad_kernel(int64_t num_pairs, int n, const double* __restrict__ gd,
                                                        const double* __restrict__ vvd, const double* __restrict__ w,
                                                        double* __restrict__ grad_w) {
  double acc[SYMPA_MAX_N];
#pragma unroll
  for (int k = 0; k < SYMPA_MAX_N; ++k) acc[k] = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < num_pairs; p += stride) {
    const double g = __ldg(gd + p);
#pragma unroll
    for (int k = 0; k < SYMPA_MAX_N; ++k)
      if (k < n) acc[k] += g * __ldg(vvd + p * n + k);
  }
#pragma unroll
  for (int k = 0; k < SYMPA_MAX_N; ++k) {
    if (k < n) {
      double v = warp_sum_d(acc[k]);
      if ((threadIdx.x & 31) == 0 && __ldg(w + k) > 0.0) atomicAdd(grad_w + k, v);
    }
  }
}

// index pairs of a block of the all-pairs distance matrix: pair t of the chunk is entry first + t of the
// row-major (row_count x num_rows) block whose first row is row_begin.  The diagonal asks for the
// next node instead (its entry is overwritten with 0 afterwards), as sympa/runner.py:148 does.
__global__ void __launch_bounds__(256) all_pairs_index_kernel(int64_t first, int64_t count, int64_t num_rows,
                                                              int64_t row_begin, longlong2* __restrict__ idx) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < count; t += stride) {
    const int64_t e = first + t;
    const int64_t r = e / num_rows;
    const int64_t j = e - r * num_rows;
    int64_t i = row_begin + r;
    if (i == j) i = (i + 1) % num_rows;
    idx[t] = make_longlong2(i, j);
  }
}

__global__ void __launch_bounds__(256) zero_diagonal_kernel(int64_t row_begin, int64_t row_count, int64_t num_rows,
                                                            double* __restrict__ out) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < row_count && row_begin + r < num_rows) out[r * num_rows + row_begin + r] = 0.0;
}

// AverageDistortionLoss (sympa/losses.py:10-19): L = sum_p | (d_p / g_p)^2 - 1 |, as one kernel forward and one
// backward instead of the five + six element-wise torch kernels of the Python expression.
__global__ void __launch_bounds__(256) distortion_loss_fwd_kernel(int64_t b, const double* __restrict__ g,
                                                                  const double* __restrict__ d, double* __restrict__ loss) {
  double acc = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < b; p += stride) {
    const double r = __ldg(d + p) / __ldg(g + p);
    acc += fabs(r * r - 1.0);
  }
  acc = warp_sum_d(acc);
  __shared__ double part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += part[w];
    atomicAdd(loss, t);
  }
}

__global__ void __launch_bounds__(256) distortion_loss_bwd_kernel(int64_t b, const double* __restrict__ g,
                                                                  const double* __restrict__ d,
                                                                  const double* __restrict__ grad_loss,
                                                                  double* __restrict__ grad_d) {
  const double go = __ldg(grad_loss);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < b; p += stride) {
    const double gi = 1.0 / __ldg(g + p);
    const double r = __ldg(d + p) * gi;
    const double e = r * r - 1.0;
    const double sg = e > 0.0 ? 1.0 : (e < 0.0 ? -1.0 : 0.0);   // torch.abs backward: sign, 0 at 0
    grad_d[p] = go * sg * 2.0 * r * gi;
  }
}

// FP64 FMA throughput probe (diagnostic: gives bench.py a MEASURED FP64 roofline denominator; the
// driver's MEASURED_PEAKS.json only has HBM and bf16 tensor peaks).  8 independent FMA chains/thread.
__global__ void __launch_bounds__(256) fp64_probe_kernel(int iters, double seed, double* __restrict__ out) {
  double a0 = seed + threadIdx.x, a1 = a0 + 1.0, a2 = a0 + 2.0, a3 = a0 + 3.0, a4 = a0 + 4.0, a5 = a0 + 5.0,
         a6 = a0 + 6.0, a7 = a0 + 7.0;
  const double m = 0.999999, c = 1e-9;
#pragma unroll 4
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c);
    a1 = fma(a1, m, c);
    a2 = fma(a2, m, c);
    a3 = fma(a3, m, c);
    a4 = fma(a4, m, c);
    a5 = fma(a5, m, c);
    a6 = fma(a6, m, c);
    a7 = fma(a7, m, c);
  }
  const double r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
  if (r == 123.456) out[0] = r;  // never true: keeps the chains alive
}

// ------------------------------------------------------------------------------------------ host
static thread_local char g_last_cuda_error[256] = "";

int check_launch() {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(g_last_cuda_error, sizeof(g_last_cuda_error), "%s", cudaGetErrorString(e));
    return SYMPA_ERR_CUDA;
  }
  return SYMPA_OK;
}

static int sm_count() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        n <= 0)
      n = 148;
    cached = n;
  }
  return cached;
}

int grid_for(int64_t work_items, int threads, int waves_cap) {
  int64_t blocks = (work_items + threads - 1) / threads;
  int64_t cap = (int64_t)sm_count() * waves_cap;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

#define SY_DECL(K)                                                                  \
  extern template int launch_pairs<K>(int, int, const PairArgs&, cudaStream_t);     \
  extern template int launch_rsgd<K>(int, const RsgdArgs&, cudaStream_t);     \
  extern template int launch_bounded_rows<K>(int, const BoundedRowsArgs&, cudaStream_t);
SY_DECL(1) SY_DECL(2) SY_DECL(3) SY_DECL(4) SY_DECL(5) SY_DECL(6) SY_DECL(7) SY_DECL(8) SY_DECL(9) SY_DECL(10)
#undef SY_DECL

static int launch_n(int n, int kind, int mode, const PairArgs& a, cudaStream_t s) {
  switch (n) {
#define SY_CASE(K) \
  case K:          \
    return launch_pairs<K>(kind, mode, a, s);
    SY_CASE(1) SY_CASE(2) SY_CASE(3) SY_CASE(4) SY_CASE(5) SY_CASE(6) SY_CASE(7) SY_CASE(8) SY_CASE(9) SY_CASE(10)
#undef SY_CASE
  }
  return SYMPA_ERR_UNSUPPORTED;
}

static int launch_bounded_rows_n(int n, int backward, const BoundedRowsArgs& a, cudaStream_t s) {
  switch (n) {
#define SY_CASE(K) \
  case K:          \
    return launch_bounded_rows<K>(backward, a, s);
    SY_CASE(1) SY_CASE(2) SY_CASE(3) SY_CASE(4) SY_CASE(5) SY_CASE(6) SY_CASE(7) SY_CASE(8) SY_CASE(9) SY_CASE(10)
#undef SY_CASE
  }
  return SYMPA_ERR_UNSUPPORTED;
}

static int launch_rsgd_n(int n, int kind, const RsgdArgs& a, cudaStream_t s) {
  switch (n) {
#define SY_CASE(K) \
  case K:          \
    return launch_rsgd<K>(kind, a, s);
    SY_CASE(1) SY_CASE(2) SY_CASE(3) SY_CASE(4) SY_CASE(5) SY_CASE(6) SY_CASE(7) SY_CASE(8) SY_CASE(9) SY_CASE(10)
#undef SY_CASE
  }
  return SYMPA_ERR_UNSUPPORTED;
}

static bool valid_common(int kind, int n, int metric, int64_t num_pairs) {
  return kind >= 0 && kind <= 2 && n >= 1 && n <= SYMPA_MAX_N && metric >= 0 && metric <= 4 && num_pairs >= 0;
}

static int point_doubles(int kind, int n) { return (kind == SYMPA_KIND_SPD ? 1 : 2) * n * n; }

// bytes of packed gradient table one scatter pass may cover (SYMPA_OPT_SCATTER_PASS_MB).  Default: one pass.
// Passes over L2-sized row ranges were built to turn the DRAM read-modify-writes of the 168 MB packed table
// (n = 4, 2^20 rows: 852 B of traffic per pair) into L2 hits, and measured SLOWER on the B200 (2^23 pairs:
// 1 pass 1.52 ms, 2 passes of 84 MB 1.81 ms, 5 passes of 34 MB 2.51 ms, 9 passes 3.99 ms): every pass walks
// all (pair, element) work items again to find the ones in range, and that walk costs more than the traffic
// it saves.  The option stays for experiments and for sympa_table_grad_scatter_rows' range logic.
static int64_t g_scatter_pass_bytes = 1ll << 46;

// scatter-add of a batch into the rows [row_begin, row_end) of the packed gradient table, in L2-sized passes
static int launch_packed_scatter(int64_t num_pairs, int per_s, int64_t num_rows, const double* grad_dist, const int64_t* idx,
                                 const double* u1, const double* u2, double* workspace, cudaStream_t s,
                                 int64_t row_begin = 0, int64_t row_end = -1, int max_sms = 0, unsigned int* tickets = nullptr) {
  if (row_end < 0) row_end = num_rows;
  const int64_t span = row_end - row_begin;
  if (span <= 0) return SYMPA_OK;
  const int64_t total = num_pairs * (int64_t)per_s;
  if (max_sms > 0 && tickets != nullptr && row_begin == 0 && row_end == num_rows) {   // SM-partitioned, for overlap
    constexpr int U = SY_SCATTER_UNROLL;
    const int grid = grid_for((int64_t)1 << 40, 256, 8);      // one full wave: 8 CTAs of 256 threads on every SM
    if (cudaMemsetAsync(tickets, 0, 2 * sizeof(unsigned int), s) != cudaSuccess) return check_launch();
    // (tickets: at most num_pairs / 256 + grid + 1 < 2^32 for any batch that fits the memory)
    scatter_packed_part_kernel<U><<<grid, 256, 0, s>>>(num_pairs, per_s, num_rows, max_sms, tickets, grad_dist, idx, u1, u2, workspace);
    return check_launch();
  }
  const int64_t table_bytes = span * (int64_t)per_s * (int64_t)sizeof(double);
  int64_t passes = (table_bytes + g_scatter_pass_bytes - 1) / g_scatter_pass_bytes;
  // a pass costs a sweep over the indices of all pairs: no more passes than the batch can pay for
  const int64_t max_passes = 1 + num_pairs / (num_rows > 0 ? num_rows : 1);
  if (passes > max_passes) passes = max_passes;
  if (passes > 16) passes = 16;
  if (passes < 1) passes = 1;
  if (passes == 1 && row_begin == 0 && row_end == num_rows) {
    constexpr int U = SY_SCATTER_UNROLL;
    const int grid = grid_for((total + U - 1) / U, 256, 32);
    if (total + (int64_t)(U + 1) * grid * 256 < (1ll << 32))
      scatter_packed_all_kernel<U, unsigned int><<<grid, 256, 0, s>>>((unsigned int)total, per_s, num_rows, grad_dist, idx, u1, u2,
                                                                     workspace);
    else
      scatter_packed_all_kernel<U, int64_t><<<grid, 256, 0, s>>>(total, per_s, num_rows, grad_dist, idx, u1, u2, workspace);
    return check_launch();
  }
  const int64_t rows_per_pass = (span + passes - 1) / passes;
  for (int64_t lo = row_begin; lo < row_end; lo += rows_per_pass) {
    const int64_t hi = lo + rows_per_pass < row_end ? lo + rows_per_pass : row_end;
    scatter_packed_table_kernel<<<grid_for(total, 256, 32), 256, 0, s>>>(total, per_s, num_rows, lo, hi, grad_dist, idx, u1, u2,
                                                                       workspace);
    const int rc = check_launch();
    if (rc) return rc;
  }
  return SYMPA_OK;
}


// check_all_points (sympa/embeddings.py:41-47 loops over the points in Python and calls the manifold's
// check_point_on_manifold on each): one thread per table row evaluates the same predicate -
//   every kind: allclose(x, x^T, atol, rtol) on each n x n block          (siegel_manifold.py:123-124)
//   upper:      det(Im z) > 0                                              (upper_half.py:93-114)
//   bounded:    allclose(A, A^H) for A = I - conj(z) z, torch's default tolerances  (bounded_domain.py:119-150)
//   spd:        eigvalsh(x) > -atol, decided as "x + atol I has a Cholesky factorisation" (geoopt)
// and the FIRST offending row wins through an atomicMin on (row << 8 | reason), which is what the reference's
// loop reports.  Rows are read once; the arithmetic is a few hundred flops per row.
__device__ __forceinline__ bool close_enough(double a, double b, double atol, double rtol) {
  return fabs(a - b) <= atol + rtol * fabs(b);     // torch.allclose; false for NaN
}
__global__ void __launch_bounds__(128) check_points_kernel(int kind, int n, int64_t num_rows, const double* __restrict__ table,
                                                           double atol, double rtol, unsigned long long* result) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int nn = n * n;
  const int per = (kind == SYMPA_KIND_SPD ? 1 : 2) * nn;
  for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < num_rows; row += stride) {
    const double* z = table + row * per;
    int reason = 0;
    for (int e = 0; e < per && reason == 0; ++e) {
      const int blk = e / nn, r = e - blk * nn, i = r / n, j = r - i * n;
      if (!close_enough(z[e], z[blk * nn + j * n + i], atol, rtol)) reason = 1;
    }
    if (reason == 0) {
      double m[SYMPA_MAX_N * SYMPA_MAX_N];
      if (kind == SYMPA_KIND_UPPER) {           // sign of det(Y): Gaussian elimination with partial pivoting
        for (int e = 0; e < nn; ++e) m[e] = z[nn + e];
        bool positive = true, zero = false;
        for (int k = 0; k < n && !zero; ++k) {
          int piv = k;
          for (int i = k + 1; i < n; ++i)
            if (fabs(m[i * n + k]) > fabs(m[piv * n + k])) piv = i;
          if (piv != k) {
            for (int j = 0; j < n; ++j) {
              const double t = m[k * n + j];
              m[k * n + j] = m[piv * n + j];
              m[piv * n + j] = t;
            }
            positive = !positive;
          }
          const double d = m[k * n + k];
          if (!(fabs(d) > 0.0)) { zero = true; break; }      // singular (or NaN): det is not > 0
          if (d < 0.0) positive = !positive;
          for (int i = k + 1; i < n; ++i) {
            const double f = m[i * n + k] / d;
            for (int j = k + 1; j < n; ++j) m[i * n + j] -= f * m[k * n + j];
          }
        }
        if (zero || !positive) reason = 2;
      } else if (kind == SYMPA_KIND_BOUNDED) {  // A = I - conj(z) z; allclose(A, A^H), rtol 1e-5, atol 1e-8
        const double* x = z;
        const double* y = z + nn;
        for (int i = 0; i < n && reason == 0; ++i)
          for (int j = 0; j <= i && reason == 0; ++j) {
            double ar = 0.0, ai = 0.0, br = 0.0, bi = 0.0;   // a = (conj(z) z)_ij, b = (conj(z) z)_ji
            for (int k = 0; k < n; ++k) {
              ar += x[i * n + k] * x[k * n + j] + y[i * n + k] * y[k * n + j];
              ai += x[i * n + k] * y[k * n + j] - y[i * n + k] * x[k * n + j];
              br += x[j * n + k] * x[k * n + i] + y[j * n + k] * y[k * n + i];
              bi += x[j * n + k] * y[k * n + i] - y[j * n + k] * x[k * n + i];
            }
            const double d = (i == j) ? 1.0 : 0.0;
            // A_ij = d - a, (A^H)_ij = conj(A_ji) = d - conj(b)
            const double pr = d - ar, pi = -ai, qr = d - br, qi = bi;
            const double diff = sqrt((pr - qr) * (pr - qr) + (pi - qi) * (pi - qi));
            if (!(diff <= 1e-8 + 1e-5 * sqrt(qr * qr + qi * qi)) || !(diff <= 1e-8 + 1e-5 * sqrt(pr * pr + pi * pi))) reason = 2;
          }
      } else {                                  // spd: Cholesky of x + atol I on the lower triangle
        for (int e = 0; e < nn; ++e) m[e] = z[e];
        for (int j = 0; j < n && reason == 0; ++j) {
          double d = m[j * n + j] + atol;
          for (int k = 0; k < j; ++k) d -= m[j * n + k] * m[j * n + k];
          if (!(d > 0.0)) { reason = 2; break; }
          const double r = 1.0 / sqrt(d);
          m[j * n + j] = d * r;
          for (int i = j + 1; i < n; ++i) {
            double v = m[i * n + j];
            for (int k = 0; k < j; ++k) v -= m[i * n + k] * m[j * n + k];
            m[i * n + j] = v * r;
          }
        }
      }
    }
    if (reason != 0) atomicMin(result, ((unsigned long long)row << 8) | (unsigned long long)reason);
  }
}

}  // namespace sympa

using namespace sympa;

extern "C" {

int sympa_version(void) { return SYMPA_ABI_VERSION; }

const char* sympa_error_string(int code) {
  switch (code) {
    case SYMPA_OK: return "ok";
    case SYMPA_ERR_BAD_ARG: return "bad argument";
    case SYMPA_ERR_UNSUPPORTED: return "unsupported kind / metric / matrix size";
    case SYMPA_ERR_CUDA: return "CUDA error";
  }
  return "unknown";
}

const char* sympa_last_cuda_error(void) { return g_last_cuda_error; }

int64_t sympa_workspace_bytes(int kind, int n, int64_t num_pairs) {
  if (kind < 0 || kind > 2 || n < 1 || n > SYMPA_MAX_N || num_pairs < 0) return -1;
  return 2 * num_pairs * (int64_t)state_doubles(kind, n) * (int64_t)sizeof(double);
}

static const int64_t kSplitChunkPairs = 32768;  // scratch per chunk stays L2-resident (n = 10: 134 MB .. n = 5: 35 MB)
static const int64_t kSplitMinPairs = 2048;     // below this the single-kernel path is used

// The three-kernel path is measured SLOWER than the single cooperative kernel in round 1 (its
// prologue / backward kernels are latency-bound at the same occupancy); it stays selectable for
// experiments and for its parity test: sympa_set_option(SYMPA_OPT_SPLIT_PATH, 1).
static int g_split_enabled = 0;
static bool uses_scratch(int kind, int n) { return g_split_enabled && kind == SYMPA_KIND_UPPER && n > SY_REG_MAX_N; }
static int64_t scratch_per_pair_bytes(int n) { return (int64_t)(5 * n * n + n) * (int64_t)sizeof(double); }
static int64_t scratch_tail_bytes(int n, int64_t num_pairs) { return num_pairs * (int64_t)(1 + n) * (int64_t)sizeof(double); }

int sympa_rsgd_step(int kind, int n, int64_t num_rows, double* table, const double* grad, double lr,
                    const double* lr_scale, unsigned long long* projected, void* stream) {
  return sympa_rsgd_step_ex(kind, n, num_rows, table, const_cast<double*>(grad), lr, lr_scale, projected, 0, stream);
}

int sympa_rsgd_step_ex(int kind, int n, int64_t num_rows, double* table, double* grad, double lr,
                       const double* lr_scale, unsigned long long* projected, int zero_grad, void* stream) {
  if (n < 1 || n > SYMPA_MAX_N) return SYMPA_ERR_UNSUPPORTED;
  if (kind != SYMPA_KIND_UPPER && kind != SYMPA_KIND_SPD && kind != SYMPA_KIND_BOUNDED) return SYMPA_ERR_UNSUPPORTED;
  if (num_rows < 0 || table == nullptr || grad == nullptr) return SYMPA_ERR_BAD_ARG;
  if (num_rows == 0) return SYMPA_OK;
  RsgdArgs a = {};
  a.num_rows = num_rows;
  a.table = table;
  a.grad = grad;
  a.lr = lr;
  a.lr_scale = lr_scale;
  a.projected = projected;
  a.zero_grad = zero_grad;
  return launch_rsgd_n(n, kind, a, (cudaStream_t)stream);
}

int64_t sympa_probe_fp64(int iters, double* out, void* stream) {
  if (iters <= 0 || out == nullptr) return -1;
  const int blocks = sm_count() * 8;
  fp64_probe_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(iters, 1.0, out);
  if (check_launch()) return -1;
  return (int64_t)blocks * 256 * 8 * 2 * (int64_t)iters;  // floating-point operations issued
}

int sympa_set_option(int option, int value) {
  if (option == SYMPA_OPT_SPLIT_PATH) {
    g_split_enabled = value != 0;
    return SYMPA_OK;
  }
  if (option == SYMPA_OPT_SCATTER_PASS_MB) {
    if (value < 1) return SYMPA_ERR_BAD_ARG;
    g_scatter_pass_bytes = (int64_t)value << 20;
    return SYMPA_OK;
  }
  return SYMPA_ERR_BAD_ARG;
}

int64_t sympa_scratch_bytes(int kind, int n, int64_t num_pairs) {
  if (kind < 0 || kind > 2 || n < 1 || n > SYMPA_MAX_N || num_pairs < 0) return -1;
  if (!uses_scratch(kind, n) || num_pairs < kSplitMinPairs) return 0;
  const int64_t cap = num_pairs < kSplitChunkPairs ? num_pairs : kSplitChunkPairs;
  return cap * scratch_per_pair_bytes(n) + scratch_tail_bytes(n, num_pairs);
}

// carve the caller's scratch: [chunk planes][dist: num_pairs][vvd: num_pairs * n]
static void setup_scratch(PairArgs* a, int kind, int n, double* scratch, int64_t scratch_bytes, bool need_tail) {
  a->scratch = nullptr;
  a->scratch_pairs = 0;
  if (scratch == nullptr || !uses_scratch(kind, n) || a->num_pairs < kSplitMinPairs) return;
  const int64_t tail = scratch_tail_bytes(n, a->num_pairs);
  if (scratch_bytes <= tail) return;
  int64_t cap = (scratch_bytes - tail) / scratch_per_pair_bytes(n);
  if (cap > a->num_pairs) cap = a->num_pairs;
  if (cap < kSplitMinPairs) return;
  a->scratch = scratch;
  a->scratch_pairs = cap;
  if (need_tail) {
    double* t = scratch + cap * (scratch_per_pair_bytes(n) / (int64_t)sizeof(double));
    if (a->dist_out == nullptr) a->dist_out = t;
    if (a->vvd_out == nullptr && a->metric == SYMPA_METRIC_WSUM) a->vvd_out = t + a->num_pairs;
  }
}

int sympa_dist_forward(int kind, int n, int metric, int64_t num_pairs, const double* z1, const double* z2,
                       const double* table, int64_t num_rows, const int64_t* idx, const double* wsum_w,
                       double* dist_out, double* vvd_out, double* saved_state, double* scratch,
                       int64_t scratch_bytes, unsigned int* status, void* stream) {
  if (!valid_common(kind, n, metric, num_pairs)) return (n < 1 || n > SYMPA_MAX_N) ? SYMPA_ERR_UNSUPPORTED : SYMPA_ERR_BAD_ARG;
  const bool mat = z1 != nullptr || z2 != nullptr;
  const bool tab = table != nullptr || idx != nullptr;
  if (mat == tab) return SYMPA_ERR_BAD_ARG;
  if (mat && (z1 == nullptr || z2 == nullptr)) return SYMPA_ERR_BAD_ARG;
  if (tab && (table == nullptr || idx == nullptr || num_rows <= 0)) return SYMPA_ERR_BAD_ARG;
  if (dist_out == nullptr) return SYMPA_ERR_BAD_ARG;
  if (metric == SYMPA_METRIC_WSUM && kind != SYMPA_KIND_SPD && wsum_w == nullptr) return SYMPA_ERR_BAD_ARG;
  if (num_pairs == 0) return SYMPA_OK;
  PairArgs a = {};
  a.num_pairs = num_pairs;
  a.z1 = z1;
  a.z2 = z2;
  a.table = table;
  a.num_rows = num_rows;
  a.idx = idx;
  a.wsum_w = wsum_w;
  a.dist_out = dist_out;
  a.vvd_out = vvd_out;
  a.status = status;
  a.metric = metric;
  if (saved_state != nullptr) {
    a.gz1 = saved_state;
    a.gz2 = saved_state + num_pairs * (int64_t)state_doubles(kind, n);
  }
  setup_scratch(&a, kind, n, scratch, scratch_bytes, false);
  return launch_n(n, kind, saved_state != nullptr ? kModeFwdSave : kModeFwd, a, (cudaStream_t)stream);
}

int sympa_dist_matrix(int kind, int n, int metric, const double* table, int64_t num_rows, int64_t row_begin,
                      int64_t row_count, const double* wsum_w, double* dist_out, int64_t* idx_workspace,
                      int64_t workspace_pairs, unsigned int* status, void* stream) {
  if (!valid_common(kind, n, metric, 0)) return (n < 1 || n > SYMPA_MAX_N) ? SYMPA_ERR_UNSUPPORTED : SYMPA_ERR_BAD_ARG;
  if (table == nullptr || dist_out == nullptr || idx_workspace == nullptr || workspace_pairs <= 0) return SYMPA_ERR_BAD_ARG;
  if (num_rows <= 0 || row_begin < 0 || row_count < 0 || row_begin + row_count > num_rows) return SYMPA_ERR_BAD_ARG;
  if (metric == SYMPA_METRIC_WSUM && kind != SYMPA_KIND_SPD && wsum_w == nullptr) return SYMPA_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t total = row_count * num_rows;
  for (int64_t first = 0; first < total; first += workspace_pairs) {
    const int64_t count = (total - first) < workspace_pairs ? (total - first) : workspace_pairs;
    all_pairs_index_kernel<<<grid_for(count, 256, 8), 256, 0, s>>>(first, count, num_rows, row_begin,
                                                                 reinterpret_cast<longlong2*>(idx_workspace));
    int rc = check_launch();
    if (rc) return rc;
    rc = sympa_dist_forward(kind, n, metric, count, nullptr, nullptr, table, num_rows, idx_workspace, wsum_w,
                            dist_out + first, nullptr, nullptr, nullptr, 0, status, stream);
    if (rc) return rc;
  }
  if (row_count > 0) {
    zero_diagonal_kernel<<<(int)((row_count + 255) / 256), 256, 0, s>>>(row_begin, row_count, num_rows, dist_out);
    return check_launch();
  }
  return SYMPA_OK;
}

int64_t sympa_average_precision_workspace_bytes(int64_t row_count, int64_t adj_entries) {
  if (row_count < 0 || adj_entries < 0) return -1;
  return (2 * row_count + 2 * adj_entries) * (int64_t)sizeof(double);
}

int sympa_average_precision(int64_t row_begin, int64_t row_count, int64_t num_cols, const double* dist,
                            const int64_t* adj_ptr, const int64_t* adj_idx, double* ap_out, void* workspace,
                            int64_t workspace_bytes, unsigned int* status, void* stream) {
  if (row_begin < 0 || row_count < 0 || num_cols <= 0 || row_begin + row_count > num_cols) return SYMPA_ERR_BAD_ARG;
  if (dist == nullptr || adj_ptr == nullptr || ap_out == nullptr || workspace == nullptr) return SYMPA_ERR_BAD_ARG;
  if (row_count > 0x7FFFFFFFll) return SYMPA_ERR_BAD_ARG;
  const int64_t cap = workspace_bytes / (int64_t)sizeof(double) / 2 - row_count;
  if (workspace_bytes < sympa_average_precision_workspace_bytes(row_count, 0) || cap < 0) return SYMPA_ERR_BAD_ARG;
  if (row_count == 0) return SYMPA_OK;
  if (adj_idx == nullptr && cap > 0) return SYMPA_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  int64_t* meta = static_cast<int64_t*>(workspace);
  double* sorted = reinterpret_cast<double*>(meta + 2 * row_count);
  unsigned long long* counts = reinterpret_cast<unsigned long long*>(sorted + cap);
  ap_prepare_kernel<<<(unsigned)row_count, SY_AP_THREADS, 0, s>>>(row_begin, num_cols, dist, adj_ptr, adj_idx, cap, meta,
                                                                   sorted, counts, status);
  int rc = check_launch();
  if (rc) return rc;
  // split each row over several CTAs until the grid is ~8 CTAs per SM, each CTA keeping >= 16 columns per thread
  const int64_t want = (int64_t)sm_count() * 8;
  int64_t splits = (want + row_count - 1) / row_count;
  const int64_t most = (num_cols + SY_AP_THREADS * 16 - 1) / (SY_AP_THREADS * 16);
  if (splits > most) splits = most;
  if (splits < 1) splits = 1;
  if (row_count * splits > 0x7FFFFFFFll) splits = 1;
  ap_count_kernel<<<(unsigned)(row_count * splits), SY_AP_THREADS, 0, s>>>(row_begin, num_cols, (int)splits, dist, adj_ptr,
                                                                           meta, sorted, counts, status);
  rc = check_launch();
  if (rc) return rc;
  ap_finish_kernel<<<(unsigned)((row_count + SY_AP_THREADS - 1) / SY_AP_THREADS), SY_AP_THREADS, 0, s>>>(
      row_begin, row_count, adj_ptr, meta, sorted, counts, ap_out);
  return check_launch();
}

int64_t sympa_hop_distances_workspace_bytes(int64_t num_nodes) {
  if (num_nodes < 0 || num_nodes > 0x7FFFFFFFll) return -1;
  return SY_HOP_HEADER_BYTES + (int64_t)SY_HOP_CTAS_PER_SM * sm_count() * num_nodes * (int64_t)sizeof(int);
}

int sympa_hop_distances(int64_t row_begin, int64_t row_count, int64_t num_nodes, const int64_t* adj_ptr,
                        const int64_t* adj_idx, int32_t* hops_out, void* workspace, int64_t workspace_bytes,
                        unsigned int* status, void* stream) {
  if (row_begin < 0 || row_count < 0 || num_nodes < 0 || num_nodes > 0x7FFFFFFFll || row_begin + row_count > num_nodes)
    return SYMPA_ERR_BAD_ARG;
  if (row_count == 0) return SYMPA_OK;
  if (adj_ptr == nullptr || adj_idx == nullptr || hops_out == nullptr || workspace == nullptr) return SYMPA_ERR_BAD_ARG;
  if (workspace_bytes < sympa_hop_distances_workspace_bytes(num_nodes)) return SYMPA_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned int* ticket = static_cast<unsigned int*>(workspace);
  int* queues = reinterpret_cast<int*>(static_cast<char*>(workspace) + SY_HOP_HEADER_BYTES);
  if (cudaMemsetAsync(ticket, 0, sizeof(unsigned int), s) != cudaSuccess) return check_launch();
  int64_t grid = (int64_t)SY_HOP_CTAS_PER_SM * sm_count();
  if (grid > row_count) grid = row_count;
  const int64_t visited_bytes = (num_nodes + 31) / 32 * (int64_t)sizeof(unsigned int);
  static_assert(SY_HOP_SMEM_VISITED_BYTES <= 48 * 1024 - 256,
                "the bitmap must leave room for the kernel's static shared memory under the 48 KB default");
  if (visited_bytes <= SY_HOP_SMEM_VISITED_BYTES)
    hop_bfs_kernel<true><<<(unsigned)grid, SY_HOP_THREADS, (size_t)visited_bytes, s>>>(
        row_begin, (int)row_count, (int)num_nodes, adj_ptr, adj_idx, hops_out, queues, ticket, status);
  else
    hop_bfs_kernel<false><<<(unsigned)grid, SY_HOP_THREADS, 0, s>>>(row_begin, (int)row_count, (int)num_nodes, adj_ptr,
                                                                    adj_idx, hops_out, queues, ticket, status);
  return check_launch();
}

int64_t sympa_sample_pairs_workspace_bytes(int64_t num_nodes) {
  if (num_nodes < 0 || num_nodes > 0x7FFFFFFFll) return -1;
  return SY_HOP_HEADER_BYTES + (int64_t)SY_HOP_CTAS_PER_SM * sm_count() * sample_slice_ints(num_nodes) * (int64_t)sizeof(int);
}

int sympa_sample_pairs(int64_t num_nodes, const int64_t* adj_ptr, const int64_t* adj_idx, int64_t num_sources,
                       const int64_t* sources, int64_t pairs_per_source, uint64_t seed, uint64_t epoch,
                       int64_t* idx_out, double* dist_out, void* workspace, int64_t workspace_bytes,
                       unsigned int* status, void* stream) {
  if (num_nodes < 0 || num_nodes > 0x7FFFFFFFll || num_sources < 0 || num_sources > 0x7FFFFFFFll || pairs_per_source < 0)
    return SYMPA_ERR_BAD_ARG;
  if (num_sources > 0 && pairs_per_source > INT64_MAX / 2 / num_sources) return SYMPA_ERR_BAD_ARG;
  if (num_sources == 0 || pairs_per_source == 0) return SYMPA_OK;
  if (adj_ptr == nullptr || adj_idx == nullptr || sources == nullptr || idx_out == nullptr || dist_out == nullptr ||
      workspace == nullptr)
    return SYMPA_ERR_BAD_ARG;
  if (workspace_bytes < sympa_sample_pairs_workspace_bytes(num_nodes)) return SYMPA_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  unsigned int* ticket = static_cast<unsigned int*>(workspace);
  int* slices = reinterpret_cast<int*>(static_cast<char*>(workspace) + SY_HOP_HEADER_BYTES);
  if (cudaMemsetAsync(ticket, 0, sizeof(unsigned int), s) != cudaSuccess) return check_launch();
  int64_t grid = (int64_t)SY_HOP_CTAS_PER_SM * sm_count();
  if (grid > num_sources) grid = num_sources;
  const int64_t visited_bytes = (num_nodes + 31) / 32 * (int64_t)sizeof(unsigned int);
  if (visited_bytes <= SY_HOP_SMEM_VISITED_BYTES)
    sample_pairs_kernel<true><<<(unsigned)grid, SY_HOP_THREADS, (size_t)visited_bytes, s>>>(
        (int)num_sources, (int)num_nodes, adj_ptr, adj_idx, sources, pairs_per_source, seed, epoch, idx_out, dist_out,
        slices, ticket, status);
  else
    sample_pairs_kernel<false><<<(unsigned)grid, SY_HOP_THREADS, 0, s>>>(
        (int)num_sources, (int)num_nodes, adj_ptr, adj_idx, sources, pairs_per_source, seed, epoch, idx_out, dist_out,
        slices, ticket, status);
  return check_launch();
}

int sympa_distortion_rows(int64_t row_begin, int64_t row_count, int64_t num_cols, const double* dist, const int32_t* hops,
                          double scale, double* sum_out, int64_t* count_out, double* max_out, double* min_out,
                          unsigned int* status, void* stream) {
  if (row_begin < 0 || row_count < 0 || num_cols < 0 || row_begin + row_count > num_cols || row_count > 0x7FFFFFFFll)
    return SYMPA_ERR_BAD_ARG;
  if (row_count == 0) return SYMPA_OK;
  if (dist == nullptr || hops == nullptr || sum_out == nullptr || count_out == nullptr || max_out == nullptr ||
      min_out == nullptr)
    return SYMPA_ERR_BAD_ARG;
  distortion_rows_kernel<<<(unsigned)row_count, SY_DISTORTION_THREADS, 0, (cudaStream_t)stream>>>(
      row_begin, num_cols, dist, hops, scale, sum_out, count_out, max_out, min_out, status);
  return check_launch();
}

int sympa_dist_backward(int kind, int n, int metric, int64_t num_pairs, const double* grad_dist,
                        const double* saved_state, double* grad_z1, double* grad_z2, double* grad_table,
                        int64_t num_rows, const int64_t* idx, const double* vvd, const double* wsum_w,
                        double* grad_wsum_w, void* stream) {
  if (!valid_common(kind, n, metric, num_pairs)) return (n < 1 || n > SYMPA_MAX_N) ? SYMPA_ERR_UNSUPPORTED : SYMPA_ERR_BAD_ARG;
  if (grad_dist == nullptr || saved_state == nullptr) return SYMPA_ERR_BAD_ARG;
  const bool mat = grad_z1 != nullptr || grad_z2 != nullptr;
  const bool tab = grad_table != nullptr;
  if (mat && (grad_z1 == nullptr || grad_z2 == nullptr)) return SYMPA_ERR_BAD_ARG;
  if (tab && (idx == nullptr || num_rows <= 0)) return SYMPA_ERR_BAD_ARG;
  if (!mat && !tab && grad_wsum_w == nullptr) return SYMPA_ERR_BAD_ARG;
  if (grad_wsum_w != nullptr && (vvd == nullptr || wsum_w == nullptr)) return SYMPA_ERR_BAD_ARG;
  if (num_pairs == 0) return SYMPA_OK;
  cudaStream_t s = (cudaStream_t)stream;
  const int per = point_doubles(kind, n);
  const int per_s = state_doubles(kind, n);
  const bool packed = state_is_packed(kind, n);
  const double* u1 = saved_state;
  const double* u2 = saved_state + num_pairs * (int64_t)per_s;
  int rc = SYMPA_OK;
  if (mat) {
    if (packed) {
      const int64_t total = num_pairs * (int64_t)per;
      scale_kernel_packed<<<grid_for(total, 256, 32), 256, 0, s>>>(total, per, per_s, n, grad_dist, u1, u2, grad_z1, grad_z2);
    } else if (per % 2 == 0) {
      const int64_t total2 = num_pairs * (int64_t)(per / 2);
      scale_kernel<<<grid_for(total2, 256, 32), 256, 0, s>>>(total2, per / 2, grad_dist, (const double2*)u1,
                                                             (const double2*)u2, (double2*)grad_z1, (double2*)grad_z2);
    } else {  // spd with odd n
      const int64_t total = num_pairs * (int64_t)per;
      scale_kernel1<<<grid_for(total, 256, 32), 256, 0, s>>>(total, per, grad_dist, u1, u2, grad_z1, grad_z2);
    }
    rc = check_launch();
    if (rc) return rc;
  }
  if (tab) {
    const int64_t total = num_pairs * (int64_t)per;
    if (packed)
      scatter_kernel_packed<<<grid_for(total, 256, 32), 256, 0, s>>>(total, per, per_s, n, num_rows, grad_dist, idx, u1, u2,
                                                                   grad_table);
    else
      scatter_kernel<<<grid_for(total, 256, 32), 256, 0, s>>>(total, per, num_rows, grad_dist, idx, u1, u2, grad_table);
    rc = check_launch();
    if (rc) return rc;
  }
  if (grad_wsum_w != nullptr && metric == SYMPA_METRIC_WSUM) {
    wsum_grad_kernel<<<grid_for(num_pairs, 256, 4), 256, 0, s>>>(num_pairs, n, grad_dist, vvd, wsum_w, grad_wsum_w);
    rc = check_launch();
  }
  return rc;
}

int sympa_bounded_rows_to_upper(int n, int64_t num_rows, const double* table, double* upper_out, unsigned int* status,
                                void* stream) {
  if (n < 1 || n > SYMPA_MAX_N) return SYMPA_ERR_UNSUPPORTED;
  if (num_rows < 0 || (num_rows > 0 && (table == nullptr || upper_out == nullptr))) return SYMPA_ERR_BAD_ARG;
  if (num_rows == 0) return SYMPA_OK;
  BoundedRowsArgs a = {};
  a.num_rows = num_rows;
  a.table = table;
  a.upper_out = upper_out;
  a.status = status;
  return launch_bounded_rows_n(n, 0, a, (cudaStream_t)stream);
}

int sympa_bounded_rows_backward(int n, int64_t num_rows, const double* table, const double* grad_upper,
                                double* grad_table, int overwrite, void* stream) {
  if (n < 1 || n > SYMPA_MAX_N) return SYMPA_ERR_UNSUPPORTED;
  if (num_rows < 0 || (num_rows > 0 && (table == nullptr || grad_upper == nullptr || grad_table == nullptr)))
    return SYMPA_ERR_BAD_ARG;
  if (num_rows == 0) return SYMPA_OK;
  BoundedRowsArgs a = {};
  a.num_rows = num_rows;
  a.table = table;
  a.grad_upper = grad_upper;
  a.grad_table = grad_table;
  a.overwrite = overwrite;
  return launch_bounded_rows_n(n, 1, a, (cudaStream_t)stream);
}

int sympa_distortion_loss_forward(int64_t num_pairs, const double* graph_dist, const double* manifold_dist,
                                  double* loss_out, void* stream) {
  if (num_pairs < 0 || loss_out == nullptr) return SYMPA_ERR_BAD_ARG;
  if (num_pairs == 0) return SYMPA_OK;
  if (graph_dist == nullptr || manifold_dist == nullptr) return SYMPA_ERR_BAD_ARG;
  distortion_loss_fwd_kernel<<<grid_for(num_pairs, 256, 8), 256, 0, (cudaStream_t)stream>>>(num_pairs, graph_dist,
                                                                                          manifold_dist, loss_out);
  return check_launch();
}

int sympa_distortion_loss_backward(int64_t num_pairs, const double* graph_dist, const double* manifold_dist,
                                   const double* grad_loss, double* grad_manifold_dist, void* stream) {
  if (num_pairs < 0) return SYMPA_ERR_BAD_ARG;
  if (num_pairs == 0) return SYMPA_OK;
  if (graph_dist == nullptr || manifold_dist == nullptr || grad_loss == nullptr || grad_manifold_dist == nullptr)
    return SYMPA_ERR_BAD_ARG;
  distortion_loss_bwd_kernel<<<grid_for(num_pairs, 256, 32), 256, 0, (cudaStream_t)stream>>>(
      num_pairs, graph_dist, manifold_dist, grad_loss, grad_manifold_dist);
  return check_launch();
}

int sympa_check_points(int kind, int n, int64_t num_rows, const double* table, double atol, double rtol,
                       unsigned long long* result, void* stream) {
  if (kind < 0 || kind > 2 || n < 1 || n > SYMPA_MAX_N) return SYMPA_ERR_UNSUPPORTED;
  if (num_rows < 0 || result == nullptr || (num_rows > 0 && table == nullptr)) return SYMPA_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaMemsetAsync(result, 0xFF, sizeof(unsigned long long), s) != cudaSuccess) return check_launch();
  if (num_rows == 0) return SYMPA_OK;
  check_points_kernel<<<grid_for(num_rows, 128, 16), 128, 0, s>>>(kind, n, num_rows, table, atol, rtol, result);
  return check_launch();
}

int64_t sympa_backward_workspace_bytes(int kind, int n, int64_t num_rows) {
  if (kind < 0 || kind > 2 || n < 1 || n > SYMPA_MAX_N || num_rows < 0) return -1;
  if (!state_is_packed(kind, n)) return 0;
  return num_rows * (int64_t)state_doubles(kind, n) * (int64_t)sizeof(double);
}

int sympa_dist_backward_table(int kind, int n, int metric, int64_t num_pairs, const double* grad_dist,
                              const double* saved_state, double* grad_table, int64_t num_rows, const int64_t* idx,
                              const double* vvd, const double* wsum_w, double* grad_wsum_w, double* workspace,
                              int64_t workspace_bytes, int overwrite, void* stream) {
  if (!valid_common(kind, n, metric, num_pairs)) return (n < 1 || n > SYMPA_MAX_N) ? SYMPA_ERR_UNSUPPORTED : SYMPA_ERR_BAD_ARG;
  if (grad_dist == nullptr || saved_state == nullptr || grad_table == nullptr || idx == nullptr || num_rows <= 0)
    return SYMPA_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  const int per = point_doubles(kind, n);
  const int per_s = state_doubles(kind, n);
  const int64_t need = sympa_backward_workspace_bytes(kind, n, num_rows);
  // the packed route pays one pass over the whole table: only when the batch covers it densely
  const bool use_ws = workspace != nullptr && need > 0 && workspace_bytes >= need && 2 * num_pairs >= num_rows;
  if (!use_ws) {
    if (overwrite && cudaMemsetAsync(grad_table, 0, (size_t)num_rows * per * sizeof(double), s) != cudaSuccess) return check_launch();
    return sympa_dist_backward(kind, n, metric, num_pairs, grad_dist, saved_state, nullptr, nullptr, grad_table, num_rows,
                               idx, vvd, wsum_w, grad_wsum_w, stream);
  }
  if (cudaMemsetAsync(workspace, 0, (size_t)need, s) != cudaSuccess) return check_launch();
  int rc = SYMPA_OK;
  if (num_pairs > 0) {
    rc = launch_packed_scatter(num_pairs, per_s, num_rows, grad_dist, idx, saved_state, saved_state + num_pairs * (int64_t)per_s,
                               workspace, s);
    if (rc) return rc;
  }
  const int64_t tot = num_rows * (int64_t)per;
  expand_table_kernel<<<grid_for(per % 2 == 0 ? tot / 2 : tot, 256, 32), 256, 0, s>>>(tot, per, per_s, n, overwrite, workspace,
                                                                                    grad_table);
  rc = check_launch();
  if (rc) return rc;
  if (grad_wsum_w != nullptr && metric == SYMPA_METRIC_WSUM && num_pairs > 0) {
    if (vvd == nullptr || wsum_w == nullptr) return SYMPA_ERR_BAD_ARG;
    wsum_grad_kernel<<<grid_for(num_pairs, 256, 4), 256, 0, s>>>(num_pairs, n, grad_dist, vvd, wsum_w, grad_wsum_w);
    rc = check_launch();
  }
  return rc;
}

int sympa_table_grad_scatter(int kind, int n, int metric, int64_t num_pairs, const double* grad_dist,
                             const double* saved_state, int64_t num_rows, const int64_t* idx, const double* vvd,
                             const double* wsum_w, double* grad_wsum_w, double* workspace, int64_t workspace_bytes,
                             void* stream) {
  if (!valid_common(kind, n, metric, num_pairs)) return (n < 1 || n > SYMPA_MAX_N) ? SYMPA_ERR_UNSUPPORTED : SYMPA_ERR_BAD_ARG;
  if (grad_dist == nullptr || saved_state == nullptr || idx == nullptr || num_rows <= 0) return SYMPA_ERR_BAD_ARG;
  const int64_t need = sympa_backward_workspace_bytes(kind, n, num_rows);
  if (need <= 0) return SYMPA_ERR_UNSUPPORTED;   // full-block saved state: use sympa_dist_backward
  if (workspace == nullptr || workspace_bytes < need) return SYMPA_ERR_BAD_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  const int per_s = state_doubles(kind, n);
  if (cudaMemsetAsync(workspace, 0, (size_t)need, s) != cudaSuccess) return check_launch();
  int rc = SYMPA_OK;
  if (num_pairs > 0) {
    rc = launch_packed_scatter(num_pairs, per_s, num_rows, grad_dist, idx, saved_state, saved_state + num_pairs * (int64_t)per_s,
                               workspace, s);
    if (rc) return rc;
    if (grad_wsum_w != nullptr && metric == SYMPA_METRIC_WSUM) {
      if (vvd == nullptr || wsum_w == nullptr) return SYMPA_ERR_BAD_ARG;
      wsum_grad_kernel<<<grid_for(num_pairs, 256, 4), 256, 0, s>>>(num_pairs, n, grad_dist, vvd, wsum_w, grad_wsum_w);
      rc = check_launch();
    }
  }
  return rc;
}

int sympa_table_grad_scatter_rows(int kind, int n, int64_t num_pairs, const double* grad_dist, const double* saved_state,
                                  int64_t num_rows, const int64_t* idx, int64_t row_begin, int64_t row_end, double* workspace,
                                  int64_t workspace_bytes, void* stream) {
  if (!valid_common(kind, n, 0, num_pairs)) return (n < 1 || n > SYMPA_MAX_N) ? SYMPA_ERR_UNSUPPORTED : SYMPA_ERR_BAD_ARG;
  if (num_rows <= 0 || row_begin < 0 || row_end < row_begin || row_end > num_rows) return SYMPA_ERR_BAD_ARG;
  const int64_t need = sympa_backward_workspace_bytes(kind, n, num_rows);
  if (workspace == nullptr || workspace_bytes < need) return SYMPA_ERR_BAD_ARG;
  if (num_pairs > 0 && (grad_dist == nullptr || saved_state == nullptr || idx == nullptr)) return SYMPA_ERR_BAD_ARG;
  if (row_end == row_begin) return SYMPA_OK;
  cudaStream_t s = (cudaStream_t)stream;
  const int per_s = state_doubles(kind, n);
  if (cudaMemsetAsync(workspace + row_begin * (int64_t)per_s, 0, (size_t)(row_end - row_begin) * per_s * sizeof(double), s) !=
      cudaSuccess)
    return check_launch();
  if (num_pairs == 0) return SYMPA_OK;
  return launch_packed_scatter(num_pairs, per_s, num_rows, grad_dist, idx, saved_state, saved_state + num_pairs * (int64_t)per_s,
                               workspace, s, row_begin, row_end);
}

int sympa_table_grad_scatter_add(int kind, int n, int64_t num_pairs, const double* grad_dist, const double* saved_state,
                                 int64_t num_rows, const int64_t* idx, double* workspace, int64_t workspace_bytes, int max_sms,
                                 unsigned int* tickets, void* stream) {
  if (!valid_common(kind, n, 0, num_pairs)) return (n < 1 || n > SYMPA_MAX_N) ? SYMPA_ERR_UNSUPPORTED : SYMPA_ERR_BAD_ARG;
  if (num_rows <= 0) return SYMPA_ERR_BAD_ARG;
  const int64_t need = sympa_backward_workspace_bytes(kind, n, num_rows);
  if (workspace == nullptr || workspace_bytes < need) return SYMPA_ERR_BAD_ARG;
  if (num_pairs == 0) return SYMPA_OK;
  if (grad_dist == nullptr || saved_state == nullptr || idx == nullptr) return SYMPA_ERR_BAD_ARG;
  const int per_s = state_doubles(kind, n);
  return launch_packed_scatter(num_pairs, per_s, num_rows, grad_dist, idx, saved_state, saved_state + num_pairs * (int64_t)per_s,
                               workspace, (cudaStream_t)stream, 0, -1, max_sms, tickets);
}

int sympa_table_grad_expand(int kind, int n, int64_t num_rows, const double* workspace, double* grad_table, int overwrite,
                            void* stream) {
  if (kind < 0 || kind > 2 || n < 1 || n > SYMPA_MAX_N) return SYMPA_ERR_UNSUPPORTED;
  if (!state_is_packed(kind, n)) return SYMPA_ERR_UNSUPPORTED;
  if (workspace == nullptr || grad_table == nullptr || num_rows <= 0) return SYMPA_ERR_BAD_ARG;
  const int per = point_doubles(kind, n);
  const int64_t tot = num_rows * (int64_t)per;
  expand_table_kernel<<<grid_for(per % 2 == 0 ? tot / 2 : tot, 256, 32), 256, 0, (cudaStream_t)stream>>>(
      tot, per, state_doubles(kind, n), n, overwrite, workspace, grad_table);
  return check_launch();
}

int sympa_distortion_step(int kind, int n, int metric, int64_t num_pairs, const double* table, int64_t num_rows,
                          const int64_t* idx, const double* graph_dist, double scale, const double* wsum_w,
                          double* grad_table, double* grad_wsum_w, double* grad_scale, double* loss_out,
                          double* dist_out, double* scratch, int64_t scratch_bytes, unsigned int* status,
                          void* stream) {
  if (!valid_common(kind, n, metric, num_pairs)) return (n < 1 || n > SYMPA_MAX_N) ? SYMPA_ERR_UNSUPPORTED : SYMPA_ERR_BAD_ARG;
  if (table == nullptr || idx == nullptr || graph_dist == nullptr || grad_table == nullptr || num_rows <= 0)
    return SYMPA_ERR_BAD_ARG;
  if (metric == SYMPA_METRIC_WSUM && kind != SYMPA_KIND_SPD && wsum_w == nullptr) return SYMPA_ERR_BAD_ARG;
  if (num_pairs == 0) return SYMPA_OK;
  PairArgs a = {};
  a.num_pairs = num_pairs;
  a.table = table;
  a.num_rows = num_rows;
  a.idx = idx;
  a.wsum_w = wsum_w;
  a.dist_out = dist_out;
  a.status = status;
  a.metric = metric;
  a.graph_dist = graph_dist;
  a.scale = scale;
  a.grad_table = grad_table;
  a.grad_wsum_w = grad_wsum_w;
  a.grad_scale = grad_scale;
  a.loss_out = loss_out;
  setup_scratch(&a, kind, n, scratch, scratch_bytes, true);
  return launch_n(n, kind, kModeStep, a, (cudaStream_t)stream);
}

}  // extern "C"
