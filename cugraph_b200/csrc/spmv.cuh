// The pull transform-reduce kernels: y[v] = init + alpha * sum_{(u->v)} x[u] * w(u,v)
// — per_v_transform_reduce_incoming_e specialised to reduce_op::plus and PageRank's e_op
// (reference cpp/include/cugraph/prims/detail/per_v_transform_reduce_e.cuh:389-885 and
// cpp/src/link_analysis/pagerank_impl.cuh:262-287), re-designed for B200:
//
//   * rows are in descending-degree order, so the degree>=32 rows are a PREFIX of the row space and
//     their edges a PREFIX of indices[]: that prefix is cut into fixed 1024-edge warp chunks
//     (edge-balanced, merge-path style: a hub row is spread over as many warps as it needs, a chunk
//     holds up to 32 whole rows).  Only row pieces that straddle a chunk boundary use atomics
//     (double, into acc_hi[row]); whole rows are stored directly.
//   * rows with degree < 32 use vertex-group-per-warp: 4/2/1 lanes per row chosen by the bin,
//     sub-warp shuffle reductions, contiguous rows => contiguous index reads.
// This is the sweep of graphs too small for the shared-memory piece stream (sweep.cuh) and of 64-bit-offset graphs, and
// the independent implementation the piece stream is compared with (cugraph_b200_debug_compare_sweeps).
//   * index / weight streams are read once with L1 no-allocate loads so that L1 keeps x[] lines;
//     row sums are accumulated in fp64 and rounded once (keeps 100-iteration PageRank within 1e-6
//     of an fp64 oracle).
#pragma once
#include "graph.cuh"

#include <cstdlib>

namespace b200 {

// device-resident loop state of one PageRank run (no per-iteration host round trip)
struct pr_state_t {
  double diff;        // sum |pr_new - pr_old| of the iteration being computed
  double dangling;    // sum of pr_new over vertices without out-edges
  double init;        // unvarying part added to every row in the CURRENT sweep
  double pers_scale;  // (dangling*alpha + 1-alpha) for the personalization scatter
  double last_diff;
  int iter;
  int done;
  unsigned ticket;  // CTAs of k_pagerank_finish that are done with this iteration (the last one resets it)
};

#ifndef B200_HOST_EMU
__device__ __forceinline__ int ld_stream(const int* p)
{
  int v;
  asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream(const float* p)
{
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ double ld_stream(const double* p)
{
  double v;
  asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
#else  // host emulation (emu/cuda_runtime.h): plain loads
inline int ld_stream(const int* p) { return *p; }
inline float ld_stream(const float* p) { return *p; }
inline double ld_stream(const double* p) { return *p; }
#endif

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------
// degree >= 32 prefix: one warp per 1024-edge chunk
// ------------------------------------------------------------------------------------------
template <typename O, typename T, bool WEIGHTED>
__global__ void __launch_bounds__(256)
k_spmv_hi(O const* __restrict__ offsets, int32_t const* __restrict__ indices, T const* __restrict__ weights,
          T const* __restrict__ x, T* __restrict__ y, int32_t const* __restrict__ row_vertex,
          int32_t const* __restrict__ chunk_first_row, int32_t n_chunks, long long nnz_hi,
          double* __restrict__ acc_hi, double alpha, pr_state_t const* __restrict__ st)
{
  if (st->done) return;
  const int lane = threadIdx.x & 31;
  const int c    = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
  if (c >= n_chunks) return;
  const double init  = st->init;
  const long long e0 = (long long)c * kWarpChunk;
  const long long e1 = (e0 + kWarpChunk < nnz_hi) ? e0 + kWarpChunk : nnz_hi;
  int r              = chunk_first_row[c];
  long long row_beg  = (long long)offsets[r];
  long long row_end  = (long long)offsets[r + 1];
  long long e        = e0;
  while (e < e1) {
    const long long seg_end = row_end < e1 ? row_end : e1;
    double acc              = 0.0;
    long long i             = e + lane;
    // 4 independent gathers in flight per lane
    for (; i + 96 < seg_end; i += 128) {
      int s0 = ld_stream(indices + i), s1 = ld_stream(indices + i + 32);
      int s2 = ld_stream(indices + i + 64), s3 = ld_stream(indices + i + 96);
      T x0 = x[s0], x1 = x[s1], x2 = x[s2], x3 = x[s3];
      if (WEIGHTED) {
        x0 *= ld_stream(weights + i);
        x1 *= ld_stream(weights + i + 32);
        x2 *= ld_stream(weights + i + 64);
        x3 *= ld_stream(weights + i + 96);
      }
      acc += ((double)x0 + (double)x1) + ((double)x2 + (double)x3);
    }
    for (; i < seg_end; i += 32) {
      T xv = x[ld_stream(indices + i)];
      if (WEIGHTED) xv *= ld_stream(weights + i);
      acc += (double)xv;
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      const bool whole = (row_beg >= e0) && (row_end <= e1);
      if (whole) {
        const int v = row_vertex ? row_vertex[r] : r;
        y[v]        = (T)(acc * alpha + init);
      } else {
        atomicAdd(acc_hi + r, acc);
      }
    }
    e = seg_end;
    if (e == row_end && e < e1) {
      ++r;
      row_beg = row_end;
      row_end = (long long)offsets[r + 1];
    }
  }
}

// rows that straddle chunk boundaries: fold the fp64 partials
template <typename T>
__global__ void k_spmv_hi_finish(int32_t const* __restrict__ split_rows, int32_t n_split, double* __restrict__ acc_hi,
                                 T* __restrict__ y, int32_t const* __restrict__ row_vertex, double alpha,
                                 pr_state_t const* __restrict__ st)
{
  if (st->done) return;
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_split) return;
  int r     = split_rows[k];
  int v     = row_vertex ? row_vertex[r] : r;
  y[v]      = (T)(acc_hi[r] * alpha + st->init);
  acc_hi[r] = 0.0;
}

// ------------------------------------------------------------------------------------------
// degree < 32: vertex-group-per-warp, group width by bin; last bin = empty rows (fill)
// ------------------------------------------------------------------------------------------
struct low_bins_t {
  int32_t row_begin[kNumSeg];    // first row of bin b (b = 0..5 -> seg[1..6]); [6] = n_rows
  int32_t block_begin[kNumSeg];  // first block of bin b; [6] = total blocks
};

// lanes per row in low bin b (degree in [16,32) [8,16) [4,8) [2,4) [1,2)): every lane owns up to 8
// edges and issues all of their loads back to back — these rows are latency-bound (offsets -> indices
// -> x is a chain of three dependent loads), so work per lane, not lanes per row, buys throughput.
__host__ __device__ __forceinline__ int low_bin_lanes(int b) { return b == 0 ? 4 : (b == 1 ? 2 : 1); }

template <typename O, typename T, bool WEIGHTED>
__global__ void __launch_bounds__(256)
k_spmv_low(O const* __restrict__ offsets, int32_t const* __restrict__ indices, T const* __restrict__ weights,
           T const* __restrict__ x, T* __restrict__ y, int32_t const* __restrict__ row_vertex, low_bins_t bins,
           double alpha, pr_state_t const* __restrict__ st)
{
  if (st->done) return;
  int b = 0;
#pragma unroll
  for (int k = 1; k < kNumSeg - 1; ++k)
    if ((int)blockIdx.x >= bins.block_begin[k]) b = k;
  const double init = st->init;
  const int blk     = blockIdx.x - bins.block_begin[b];
  if (b == kNumSeg - 2) {  // empty rows
    int r = bins.row_begin[b] + blk * 256 + threadIdx.x;
    if (r < bins.row_begin[b + 1]) y[row_vertex ? row_vertex[r] : r] = (T)init;
    return;
  }
  const int g   = low_bin_lanes(b);
  const int sub = threadIdx.x & (g - 1);
  const int r   = bins.row_begin[b] + blk * (256 / g) + (threadIdx.x / g);
  double acc    = 0.0;
  const bool in = r < bins.row_begin[b + 1];
  if (in) {
    const long long lo = (long long)offsets[r], hi = (long long)offsets[r + 1];
    constexpr int kR = 8;  // degree < 32 and g in {4,2,1} => at most 8 edges per lane
    int c[kR];
    T wv[kR];
#pragma unroll
    for (int k = 0; k < kR; ++k) {
      const long long e = lo + sub + (long long)k * g;
      c[k]              = 0;
      wv[k]             = (T)0;
      if (e < hi) {
        // these loads allocate in L1: a lane walks 4..32 consecutive bytes of its row, so the sectors are re-used by its
        // next loads (measured: sweep 0.470 -> 0.456 ms on RMAT-24 against streaming loads)
        c[k]  = __ldg(indices + e);
        wv[k] = WEIGHTED ? __ldg(weights + e) : (T)1;
      }
    }
    T v[kR];
#pragma unroll
    for (int k = 0; k < kR; ++k) v[k] = x[c[k]] * wv[k];
    acc = (((double)v[0] + (double)v[1]) + ((double)v[2] + (double)v[3])) +
          (((double)v[4] + (double)v[5]) + ((double)v[6] + (double)v[7]));
  }
  for (int o = g >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (in && sub == 0) y[row_vertex ? row_vertex[r] : r] = (T)(acc * alpha + init);
}

// ------------------------------------------------------------------------------------------
// host-side launcher of one full sweep
// ------------------------------------------------------------------------------------------
inline low_bins_t make_low_bins(csx_t const& c)
{
  low_bins_t b{};
  int blocks = 0;
  for (int k = 0; k < kNumSeg - 1; ++k) {
    b.row_begin[k]   = c.seg[k];
    b.block_begin[k] = blocks;
    int rows         = c.seg[k + 1] - c.seg[k];
    int per_block    = (k == kNumSeg - 2) ? 256 : 256 / low_bin_lanes(k);
    blocks += (rows + per_block - 1) / per_block;
  }
  b.row_begin[kNumSeg - 1]   = c.seg[kNumSeg];
  b.block_begin[kNumSeg - 1] = blocks;
  return b;
}

template <typename O, typename T>
void launch_pull_sweep(handle_impl const& h, csx_t const& c, T const* x, T* y, double* acc_hi, double alpha,
                       pr_state_t const* st, bool use_weights = true)
{
  O const* off        = c.offsets.as<O>();
  int32_t const* idx  = c.indices.as<int32_t>();
  T const* w          = use_weights ? c.weights.as<T>() : nullptr;  // HITS sums plain neighbour values on a weighted graph too
  int32_t const* rv   = c.row_vertex.as<int32_t>();
  const bool weighted = (w != nullptr);
  if (c.n_chunks > 0) {
    int grid = (c.n_chunks + kWarpsPerCta - 1) / kWarpsPerCta;
    if (weighted)
      B200_LAUNCH(h, (k_spmv_hi<O, T, true>), grid, 256, 0, off, idx, w, x, y, rv, c.chunk_first_row.as<int32_t>(),
                  c.n_chunks, (long long)c.nnz_hi, acc_hi, alpha, st);
    else
      B200_LAUNCH(h, (k_spmv_hi<O, T, false>), grid, 256, 0, off, idx, w, x, y, rv, c.chunk_first_row.as<int32_t>(),
                  c.n_chunks, (long long)c.nnz_hi, acc_hi, alpha, st);
    if (c.n_split > 0)
      B200_LAUNCH(h, (k_spmv_hi_finish<T>), (c.n_split + 255) / 256, 256, 0, c.split_rows.as<int32_t>(), c.n_split,
                  acc_hi, y, rv, alpha, st);
  }
  low_bins_t bins = make_low_bins(c);
  int lblocks     = bins.block_begin[kNumSeg - 1];
  if (lblocks > 0) {
    if (weighted)
      B200_LAUNCH(h, (k_spmv_low<O, T, true>), lblocks, 256, 0, off, idx, w, x, y, rv, bins, alpha, st);
    else
      B200_LAUNCH(h, (k_spmv_low<O, T, false>), lblocks, 256, 0, off, idx, w, x, y, rv, bins, alpha, st);
  }
}

}  // namespace b200
