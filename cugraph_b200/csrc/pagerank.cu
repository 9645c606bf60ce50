// PageRank on one B200 + its C-ABI entry points.
// Replaces cpp/src/link_analysis/pagerank_impl.cuh:40-330 (driver) and cpp/src/c_api/pagerank.cpp.
//
// Per iteration the reference runs ~6 V-sized thrust passes and 2 blocking scalar read-backs
// (pagerank_impl.cuh:225-318).  Here an iteration is: pull sweep (spmv.cuh) -> [personalization
// scatter] -> ONE fused vertex pass (diff, dangling sum, next x = pr/out_w) -> 1-thread finalize that
// advances the device-resident loop state; on the piece stream without personalization everything after the sweep is one
// kernel (k_pagerank_finish).  The host enqueues iterations in batches and only reads the
// `done` flag between batches; kernels of iterations past convergence are no-ops, so the iteration
// count and result are exactly those of a check-every-iteration loop.
#include "sweep.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>

namespace b200 {
namespace {

constexpr int kBlock = 256;
inline int grid_for(int64_t n) { return (int)std::min<int64_t>(std::max<int64_t>((n + kBlock - 1) / kBlock, 1), 1 << 22); }

template <typename T>
__global__ void k_fill(T* a, int32_t n, T v)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = v;
}

__global__ void k_out_degree(int32_t const* __restrict__ indices, long long nnz, int32_t* __restrict__ deg)
{
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nnz; i += (long long)gridDim.x * blockDim.x)
    atomicAdd(deg + indices[i], 1);
}

template <typename T>
__global__ void k_out_weight(int32_t const* __restrict__ indices, T const* __restrict__ w, long long nnz, double* __restrict__ sums)
{
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nnz; i += (long long)gridDim.x * blockDim.x)
    atomicAdd(sums + indices[i], (double)w[i]);
}

template <typename S, typename T>
__global__ void k_cast(S const* in, int32_t n, T* out)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (T)in[i];
}

__device__ __forceinline__ double block_sum(double v, double* smem)
{
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < 32) {
    t = (threadIdx.x < (blockDim.x >> 5)) ? smem[threadIdx.x] : 0.0;
    t = warp_sum(t);
  }
  __syncthreads();
  return t;  // valid in warp 0
}

// fused vertex pass: diff += |new-old| ; dangling += new where out_w==0 ; x = new / (out_w or 1)
template <typename T>
__global__ void __launch_bounds__(kBlock)
k_vertex_pass(T const* __restrict__ pr_new, T const* __restrict__ pr_old, T const* __restrict__ out_w,
              T* __restrict__ x, int32_t n, pr_state_t* __restrict__ st)
{
  if (st->done) return;
  __shared__ double smem[8];
  double diff = 0.0, dang = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    T nv = pr_new[i];
    T ow = out_w[i];
    if (pr_old) diff += fabs((double)nv - (double)pr_old[i]);
    if (ow == (T)0) dang += (double)nv;
    x[i] = (ow == (T)0) ? nv : nv / ow;
  }
  diff = block_sum(diff, smem);
  dang = block_sum(dang, smem);
  if (threadIdx.x == 0) {
    if (pr_old) atomicAdd(&st->diff, diff);
    atomicAdd(&st->dangling, dang);
  }
}

// advance the loop state (pagerank_impl.cuh:256-259, 320-329) from the iteration's diff and dangling sums
__device__ __forceinline__ void advance_state(pr_state_t* st, double diff, double dangling, double alpha, double epsilon,
                                              int n_vertices, int personalized, int count_iteration, int max_iterations)
{
  double base    = dangling * alpha + (1.0 - alpha);
  st->init       = personalized ? 0.0 : base / (double)n_vertices;
  st->pers_scale = base;
  if (count_iteration) {
    st->iter += 1;
    st->last_diff = diff;
    if (diff < epsilon || st->iter >= max_iterations) st->done = 1;
  }
  st->diff     = 0.0;
  st->dangling = 0.0;
}

__global__ void k_finalize(pr_state_t* st, double alpha, double epsilon, int n_vertices, int personalized,
                           int count_iteration, int max_iterations)
{
  if (st->done) return;
  advance_state(st, st->diff, st->dangling, alpha, epsilon, n_vertices, personalized, count_iteration, max_iterations);
}

template <typename T> struct vec2_of;
template <> struct vec2_of<float> { using type = float2; };
template <> struct vec2_of<double> { using type = double2; };

// The rest of a non-personalized PageRank iteration after k_sweep, in one pass over the rows (= vertices: the pull view has
// no row_vertex): pr_new = acc * alpha + init, x = pr_new / out_w (pr_new where out_w == 0), diff += |pr_new - pr_old|,
// dangling += pr_new where out_w == 0; clears the accumulators and the sweep's cursors.  The last CTA to finish (a ticket)
// advances the loop state as k_finalize does.  This is k_sweep_finish + k_vertex_pass + k_finalize without the round trip of
// pr_new through memory and without two launches per iteration.  Rows are read as in k_sweep_finish (a warp tile is
// kPrSteps steps of 64 consecutive rows, lane = two rows, every load of a tile issued before the first use); the grid is a
// few CTAs per SM, all resident, that stride over the tiles, so that only those few CTAs add their sums to the state and take a ticket.
template <typename T>
constexpr int pr_steps() { return 16 / (int)sizeof(T); }  // 4 (float) / 2 (double): the registers of 3 CTAs per SM
constexpr int kPrCtasPerSm = 3;

template <typename T>
__global__ void __launch_bounds__(256, kPrCtasPerSm)  // all CTAs of the grid resident at once
k_pagerank_finish(double* __restrict__ acc, int n_cov, int n_rows, T* __restrict__ pr_new, T const* __restrict__ pr_old,
                  T const* __restrict__ out_w, T* __restrict__ x, int* __restrict__ cursor, int n_phases, double alpha,
                  double epsilon, int max_iterations, pr_state_t* __restrict__ st)
{
  using T2 = typename vec2_of<T>::type;
  constexpr int kPrSteps = pr_steps<T>();
  __shared__ double s_red[2][8];
  if (st->done) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_phases; i += gridDim.x * blockDim.x) cursor[i] = 0;
  const int lane    = threadIdx.x & 31;
  const int n_warps = gridDim.x * (blockDim.x >> 5);
  const int n_tiles = (n_rows + 64 * kPrSteps - 1) / (64 * kPrSteps);
  const double init = st->init;
  double diff = 0.0, dang = 0.0;
  for (int tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); tile < n_tiles; tile += n_warps) {
    const int base = tile * (64 * kPrSteps) + 2 * lane;  // first of this lane's two rows in step 0
    double2 q[kPrSteps];
    T2 old[kPrSteps], ow[kPrSteps];
#pragma unroll
    for (int k = 0; k < kPrSteps; ++k) {
      const int r = base + 64 * k;
      q[k]        = make_double2(0.0, 0.0);
      if (r + 1 < n_cov) q[k] = *reinterpret_cast<double2 const*>(acc + r);
      else if (r < n_cov) q[k].x = acc[r];
      old[k] = T2{(T)0, (T)0};
      ow[k]  = T2{(T)0, (T)0};
      if (r + 1 < n_rows) {
        old[k] = *reinterpret_cast<T2 const*>(pr_old + r);
        ow[k]  = *reinterpret_cast<T2 const*>(out_w + r);
      } else if (r < n_rows) {
        old[k].x = pr_old[r];
        ow[k].x  = out_w[r];
      }
    }
#pragma unroll
    for (int k = 0; k < kPrSteps; ++k) {
      const int r = base + 64 * k;
      if (r + 1 < n_cov) *reinterpret_cast<double2*>(acc + r) = make_double2(0.0, 0.0);
      else if (r < n_cov) acc[r] = 0.0;
      if (r >= n_rows) continue;
      const T v0 = (T)(q[k].x * alpha + init), v1 = (T)(q[k].y * alpha + init);
      const T x0 = (ow[k].x == (T)0) ? v0 : v0 / ow[k].x, x1 = (ow[k].y == (T)0) ? v1 : v1 / ow[k].y;
      diff += fabs((double)v0 - (double)old[k].x);
      if (ow[k].x == (T)0) dang += (double)v0;
      if (r + 1 < n_rows) {
        diff += fabs((double)v1 - (double)old[k].y);
        if (ow[k].y == (T)0) dang += (double)v1;
        *reinterpret_cast<T2*>(pr_new + r) = T2{v0, v1};
        *reinterpret_cast<T2*>(x + r)      = T2{x0, x1};
      } else {
        pr_new[r] = v0;
        x[r]      = x0;
      }
    }
  }
  diff = warp_sum(diff);
  dang = warp_sum(dang);
  if (lane == 0) {
    s_red[0][threadIdx.x >> 5] = diff;
    s_red[1][threadIdx.x >> 5] = dang;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double d = 0.0, g = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
      d += s_red[0][w];
      g += s_red[1][w];
    }
    atomicAdd(&st->diff, d);
    atomicAdd(&st->dangling, g);
    __threadfence();  // the sums are visible before the ticket that counts them
    if (atomicAdd(&st->ticket, 1u) == gridDim.x - 1) {
      __threadfence();
      volatile pr_state_t const* vs = st;  // every CTA's sums, not a cached copy
      const double sum_diff = vs->diff, sum_dang = vs->dangling;
      advance_state(st, sum_diff, sum_dang, alpha, epsilon, n_rows, 0, 1, max_iterations);
      st->ticket = 0;
    }
  }
}

template <typename T>
__global__ void k_personalize(int32_t const* __restrict__ pv, T const* __restrict__ pvals, int32_t n, double pers_sum,
                              T* __restrict__ y, pr_state_t const* __restrict__ st)
{
  if (st->done) return;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[pv[i]] = (T)((double)y[pv[i]] + st->pers_scale * ((double)pvals[i] / pers_sum));
}

template <typename T>
__global__ void k_sum(T const* a, int32_t n, double* out)
{
  __shared__ double smem[8];
  double s = 0.0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) s += (double)a[i];
  s = block_sum(s, smem);
  if (threadIdx.x == 0) atomicAdd(out, s);
}

template <typename T>
__global__ void k_count_negative(T const* a, int64_t n, int* out)
{
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (a[i] < (T)0) atomicAdd(out, 1);
}

// ---- debug: compare the configured sweep with the plain reference sweep, row by row
template <typename T>
__global__ void k_fill_pattern(T* x, int32_t n)
{
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = (T)(0.5 + (double)((unsigned)(i * 2654435761u) >> 16) / 65536.0);
}

// packed (relative difference bits << 32 | row): atomicMax keeps the worst row of each class
template <typename O, typename T>
__global__ void k_compare_rows(O const* __restrict__ off, int32_t const* __restrict__ row_vertex, T const* __restrict__ a,
                               T const* __restrict__ b, int32_t n_rows, int32_t n_hi, double tol,
                               unsigned long long* __restrict__ worst /*[2]*/, unsigned long long* __restrict__ n_bad /*[2]*/)
{
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  const int v        = row_vertex ? row_vertex[r] : r;
  const double va = (double)a[v], vb = (double)b[v];
  const double den   = fmax(fabs(va), 1e-300);
  const float rel    = (float)fmin(fabs(va - vb) / den, 1e30);
  const int cls      = r < n_hi ? 0 : 1;
  atomicMax(worst + cls, ((unsigned long long)__float_as_uint(rel) << 32) | (unsigned)r);
  if (rel > tol) atomicAdd(n_bad + cls, 1ull);
  (void)off;
}

struct pr_args {
  device_array_view_impl const* pre_v{nullptr};
  device_array_view_impl const* pre_w{nullptr};
  device_array_view_impl const* init_v{nullptr};
  device_array_view_impl const* init_val{nullptr};
  device_array_view_impl const* pers_v{nullptr};
  device_array_view_impl const* pers_val{nullptr};
  double alpha{0.85};
  double epsilon{1e-5};
  size_t max_iterations{100};
  bool expensive{false};
};

template <typename T>
void pagerank_typed(handle_impl const& h, graph_impl& g, pr_args const& a, centrality_result_impl& res)
{
  phase_trace tr(h);
  const int32_t nv = g.n_vertices;
  // argument checks of pagerank_impl.cuh:79-88
  B200_EXPECTS(a.alpha >= 0.0 && a.alpha <= 1.0, CUGRAPH_UNKNOWN_ERROR, "Invalid input argument: alpha should be in [0.0, 1.0].");
  B200_EXPECTS(a.epsilon >= 0.0, CUGRAPH_UNKNOWN_ERROR, "Invalid input argument: epsilon should be non-negative.");
  if (nv == 0) {
    res.vertices   = new device_array_impl{dbuf(0, h.stream), 0, g.vertex_type};
    res.values     = new device_array_impl{dbuf(0, h.stream), 0, g.weight_type};
    res.iterations = 0;
    res.converged  = true;
    return;
  }
  csx_t const& c = pull_view(h, g);
  B200_EXPECTS(c.degree_sorted, CUGRAPH_UNKNOWN_ERROR, "internal: pull view is not binned");
  const bool weighted = g.weighted;

  // out-weight sums (pagerank_impl.cuh:180-198).  A property of the graph: computed once per graph
  // (the reference recomputes it on every call with a push-model prim, one atomic per edge).
  dbuf out_w_user;
  T const* out_w = nullptr;
  if (a.pre_w) {
    out_w_user = collect_vertex_values<T>(h, g, a.pre_v, a.pre_w, (T)0);
    out_w      = out_w_user.as<T>();
  } else {
    if (c.out_w.data() == nullptr) {
      dbuf ow = make_dbuf<T>(nv, h.stream);
      if (weighted) {
        dbuf sums = make_dbuf<double>(nv, h.stream);
        CUDA_TRY(cudaMemsetAsync(sums.data(), 0, sizeof(double) * nv, h.stream));
        if (c.nnz > 0)
          B200_LAUNCH(h, (k_out_weight<T>), std::min(grid_for(c.nnz), 148 * 16), kBlock, 0, c.indices.as<int32_t>(),
                      c.weights.as<T>(), (long long)c.nnz, sums.as<double>());
        B200_LAUNCH(h, (k_cast<double, T>), grid_for(nv), kBlock, 0, sums.as<double>(), nv, ow.as<T>());
      } else {
        dbuf deg = make_dbuf<int32_t>(nv, h.stream);
        CUDA_TRY(cudaMemsetAsync(deg.data(), 0, sizeof(int32_t) * nv, h.stream));
        if (c.nnz > 0)
          B200_LAUNCH(h, k_out_degree, std::min(grid_for(c.nnz), 148 * 16), kBlock, 0, c.indices.as<int32_t>(),
                      (long long)c.nnz, deg.as<int32_t>());
        B200_LAUNCH(h, (k_cast<int32_t, T>), grid_for(nv), kBlock, 0, deg.as<int32_t>(), nv, ow.as<T>());
      }
      sync(h);
      c.out_w = std::move(ow);
    }
    out_w = c.out_w.as<T>();
  }
  tr.mark("pagerank: pull view + out-weights");
  if (a.expensive && weighted && c.nnz > 0) {
    dbuf neg = make_dbuf<int>(1, h.stream);
    CUDA_TRY(cudaMemsetAsync(neg.data(), 0, sizeof(int), h.stream));
    B200_LAUNCH(h, (k_count_negative<T>), std::min(grid_for(c.nnz), 148 * 16), kBlock, 0, c.weights.as<T>(), c.nnz, neg.as<int>());
    int hneg = 0;
    CUDA_TRY(cudaMemcpyAsync(&hneg, neg.data(), sizeof(int), cudaMemcpyDeviceToHost, h.stream));
    sync(h);
    B200_EXPECTS(hneg == 0, CUGRAPH_UNKNOWN_ERROR, "Invalid input argument: input edge weights should have non-negative values.");
  }

  // personalization (pagerank_impl.cuh:200-214): ids -> internal, sum must be positive
  dbuf pers_idx, pers_vals;
  int32_t n_pers  = 0;
  double pers_sum = 0.0;
  if (a.pers_v) {
    B200_EXPECTS(a.pers_val && a.pers_v->size == a.pers_val->size, CUGRAPH_UNKNOWN_ERROR,
                 "Invalid input argument: if personalization.has_value() is true, the size of vertices and values should match");
    B200_EXPECTS(a.pers_v->size > 0, CUGRAPH_UNKNOWN_ERROR,
                 "Invalid input argument: if personalizations.has_value() is true, the input personalization vector size should not be 0.");
    n_pers   = (int32_t)a.pers_v->size;
    pers_idx = make_dbuf<int32_t>(n_pers, h.stream);
    ext_to_int(h, g, a.pers_v->data, n_pers, pers_idx.as<int32_t>());
    dbuf bad = make_dbuf<int>(1, h.stream);
    CUDA_TRY(cudaMemsetAsync(bad.data(), 0, sizeof(int), h.stream));
    B200_LAUNCH(h, (k_count_negative<int32_t>), grid_for(n_pers), kBlock, 0, pers_idx.as<int32_t>(), (int64_t)n_pers, bad.as<int>());
    dbuf dsum = make_dbuf<double>(1, h.stream);
    CUDA_TRY(cudaMemsetAsync(dsum.data(), 0, sizeof(double), h.stream));
    B200_LAUNCH(h, (k_sum<T>), std::min(grid_for(n_pers), 1024), kBlock, 0, (T const*)a.pers_val->data, n_pers, dsum.as<double>());
    int hbad = 0;
    CUDA_TRY(cudaMemcpyAsync(&hbad, bad.data(), sizeof(int), cudaMemcpyDeviceToHost, h.stream));
    CUDA_TRY(cudaMemcpyAsync(&pers_sum, dsum.data(), sizeof(double), cudaMemcpyDeviceToHost, h.stream));
    sync(h);
    B200_EXPECTS(hbad == 0, CUGRAPH_INVALID_INPUT, "Invalid input argument: peresonalization vertices have invalid vertex IDs.");
    B200_EXPECTS(pers_sum > 0.0, CUGRAPH_UNKNOWN_ERROR, "Invalid input argument: sum of personalization valuese should be positive.");
  }

  // state
  dbuf pr_a = make_dbuf<T>(nv, h.stream), pr_b = make_dbuf<T>(nv, h.stream);
  dbuf x    = make_dbuf<T>(padded_x_elems(nv, sizeof(T)), h.stream);  // whole smem slices are TMA-copied
  CUDA_TRY(cudaMemsetAsync(x.data(), 0, padded_x_elems(nv, sizeof(T)) * sizeof(T), h.stream));  // zeros behind nv
  dbuf acc_hi = make_dbuf<double>(acc_rows(c), h.stream);
  CUDA_TRY(cudaMemsetAsync(acc_hi.data(), 0, sizeof(double) * acc_rows(c), h.stream));
  dbuf state = make_dbuf<pr_state_t>(1, h.stream);
  CUDA_TRY(cudaMemsetAsync(state.data(), 0, sizeof(pr_state_t), h.stream));
  pr_state_t* st = state.as<pr_state_t>();

  if (a.init_val) {
    // the C API copies the guess as-is (cpp/src/c_api/pagerank.cpp:179-203, no normalisation)
    dbuf guess = collect_vertex_values<T>(h, g, a.init_v, a.init_val, (T)0);
    CUDA_TRY(cudaMemcpyAsync(pr_a.data(), guess.data(), sizeof(T) * nv, cudaMemcpyDeviceToDevice, h.stream));
    sync(h);
  } else {
    B200_LAUNCH(h, (k_fill<T>), grid_for(nv), kBlock, 0, pr_a.as<T>(), nv, (T)((T)1 / (T)nv));
  }

  tr.mark("pagerank: state setup");
  const int vgrid = std::min(grid_for(nv), h.sm_count * 8);
  const int max_it = (int)std::min<size_t>(a.max_iterations, 0x7fffffff);
  // prologue: x and dangling sum of the starting vector, init for sweep 1
  B200_LAUNCH(h, (k_vertex_pass<T>), vgrid, kBlock, 0, pr_a.as<T>(), (T const*)nullptr, out_w, x.as<T>(), nv, st);
  B200_LAUNCH(h, k_finalize, 1, 1, 0, st, a.alpha, a.epsilon, nv, n_pers > 0 ? 1 : 0, 0, max_it);

  T* cur = pr_a.as<T>();
  T* nxt = pr_b.as<T>();
  pr_state_t* hst = reinterpret_cast<pr_state_t*>(h.pinned);
  int enqueued    = 0;
  int iters       = 0;
  const int batch = (a.epsilon > 0.0) ? 8 : 64;
  if (max_it == 0) {
    // the reference's loop body runs at least once (pagerank_impl.cuh:224-327: test after iter++)
  }
  // Non-personalized PageRank on the piece stream, rows = vertices (a graph stored transposed): k_sweep + k_pagerank_finish.
  // Personalization scatters into pr_new between the sweep and the vertex pass, and with row_vertex the vertex-order streams
  // would be gathered through it; those take the general path.
  sweep_layout_t const* L = (!c.offs64 && n_pers == 0 && c.row_vertex.data() == nullptr && c.n_rows == nv)
                              ? sweep_layout(h, c, nv, sizeof(T)) : nullptr;
  const int fin_grid = std::max(std::min(ceil_div(nv, 64 * pr_steps<T>() * 8), h.sm_count * kPrCtasPerSm), 1);
  while (true) {
    int todo = std::min(batch, std::max(max_it, 1) - enqueued);
    for (int k = 0; k < todo; ++k) {
      if (L) {
        launch_sweep_pieces<T>(h, *L, x.as<T>(), acc_hi.as<double>(), st);
        B200_LAUNCH(h, (k_pagerank_finish<T>), fin_grid, 256, 0, acc_hi.as<double>(), L->n_cov, nv, nxt,
                    (T const*)cur, out_w, x.as<T>(), L->cursor.as<int>(), L->n_phases, a.alpha, a.epsilon, max_it, st);
      } else {
        if (c.offs64) launch_pull_sweep<int64_t, T>(h, c, x.as<T>(), nxt, acc_hi.as<double>(), a.alpha, st);
        else launch_pull_sweep_auto<int32_t, T>(h, c, nv, x.as<T>(), nxt, acc_hi.as<double>(), a.alpha, st);
        if (n_pers > 0)
          B200_LAUNCH(h, (k_personalize<T>), grid_for(n_pers), kBlock, 0, pers_idx.as<int32_t>(), (T const*)a.pers_val->data,
                      n_pers, pers_sum, nxt, st);
        B200_LAUNCH(h, (k_vertex_pass<T>), vgrid, kBlock, 0, nxt, cur, out_w, x.as<T>(), nv, st);
        B200_LAUNCH(h, k_finalize, 1, 1, 0, st, a.alpha, a.epsilon, nv, n_pers > 0 ? 1 : 0, 1, max_it);
      }
      std::swap(cur, nxt);
      ++enqueued;
    }
    check_last("pagerank iteration");
    CUDA_TRY(cudaMemcpyAsync(hst, st, sizeof(pr_state_t), cudaMemcpyDeviceToHost, h.stream));
    sync(h);
    iters = hst->iter;
    if (hst->done || enqueued >= std::max(max_it, 1)) break;
  }
  tr.mark("pagerank: iterations (+ layout staging on the first call)");
  // after `iters` real iterations the newest vector sits in pr_a when iters is even, pr_b when odd
  T* final_pr = (iters % 2 == 0) ? pr_a.as<T>() : pr_b.as<T>();

  res.vertices   = new device_array_impl{reported_vertices(h, g), (size_t)nv, g.vertex_type};
  res.values     = new device_array_impl{to_reported_order(h, g, final_pr, sizeof(T)), (size_t)nv, g.weight_type};
  res.iterations = (size_t)iters;
  res.converged  = (size_t)iters < a.max_iterations;  // pagerank_impl.cuh:329
  sync(h);
  tr.mark("pagerank: result gather");
}

cugraph_error_code_t pagerank_entry(const cugraph_resource_handle_t* handle, cugraph_graph_t* graph, pr_args a,
                                    bool require_convergence, cugraph_centrality_result_t** result,
                                    cugraph_error_t** error)
{
  return guarded(error, [&] {
    auto const& h = H(handle);
    auto* g       = G(graph);
    B200_EXPECTS(result != nullptr, CUGRAPH_INVALID_INPUT, "result out-pointer is NULL");
    *result = nullptr;
    // type checks of cpp/src/c_api/pagerank.cpp:262-293
    if (a.pre_v) {
      B200_EXPECTS(a.pre_v->type == g->vertex_type, CUGRAPH_INVALID_INPUT,
                   "vertex type of graph and precomputed_vertex_out_weight_vertices must match");
      B200_EXPECTS(a.pre_w && a.pre_w->type == g->weight_type, CUGRAPH_INVALID_INPUT,
                   "vertex type of graph and precomputed_vertex_out_weight_sums must match");
    }
    if (a.init_v) {
      B200_EXPECTS(a.init_v->type == g->vertex_type, CUGRAPH_INVALID_INPUT,
                   "vertex type of graph and initial_guess_vertices must match");
      B200_EXPECTS(a.init_val && a.init_val->type == g->weight_type, CUGRAPH_INVALID_INPUT,
                   "vertex type of graph and initial_guess_values must match");
    }
    if (a.pers_v) {
      B200_EXPECTS(a.pers_v->type == g->vertex_type, CUGRAPH_INVALID_INPUT,
                   "vertex type of graph and personalization_vector must match");
      B200_EXPECTS(a.pers_val && a.pers_val->type == g->weight_type, CUGRAPH_INVALID_INPUT,
                   "vertex type of graph and personalization_vector must match");
    }
    if (!a.pre_w) a.pre_v = nullptr;
    if (!a.init_val) a.init_v = nullptr;
    auto res = std::make_unique<centrality_result_impl>();
    if (g->mg) {
      mg_pagerank(h, *g, mg_pr_args{a.alpha, a.epsilon, a.max_iterations}, *res);
    } else if (g->weight_type == FLOAT32) {
      pagerank_typed<float>(h, *g, a, *res);
    } else {
      pagerank_typed<double>(h, *g, a, *res);
    }
    bool converged = res->converged;
    *result        = reinterpret_cast<cugraph_centrality_result_t*>(res.release());
    // cpp/src/c_api/pagerank.cpp:306-313: the result object is still returned
    B200_EXPECTS(!require_convergence || converged, CUGRAPH_UNKNOWN_ERROR, "PageRank failed to converge.");
  });
}

}  // namespace

}  // namespace b200

using namespace b200;

extern "C" {

cugraph_type_erased_device_array_view_t* cugraph_centrality_result_get_vertices(cugraph_centrality_result_t* result)
{
  auto* r = reinterpret_cast<centrality_result_impl*>(result);
  return reinterpret_cast<cugraph_type_erased_device_array_view_t*>(r->vertices->new_view());
}

cugraph_type_erased_device_array_view_t* cugraph_centrality_result_get_values(cugraph_centrality_result_t* result)
{
  auto* r = reinterpret_cast<centrality_result_impl*>(result);
  return reinterpret_cast<cugraph_type_erased_device_array_view_t*>(r->values->new_view());
}

size_t cugraph_centrality_result_get_num_iterations(cugraph_centrality_result_t* result)
{
  return reinterpret_cast<centrality_result_impl*>(result)->iterations;
}

bool_t cugraph_centrality_result_converged(cugraph_centrality_result_t* result)
{
  return reinterpret_cast<centrality_result_impl*>(result)->converged ? TRUE : FALSE;
}

void cugraph_centrality_result_free(cugraph_centrality_result_t* result)
{
  if (!result) return;
  auto* r = reinterpret_cast<centrality_result_impl*>(result);
  delete r->vertices;
  delete r->values;
  delete r;
}

#define PR_ARGS_COMMON                                                                          \
  pr_args a;                                                                                    \
  a.pre_v          = V(precomputed_vertex_out_weight_vertices);                                 \
  a.pre_w          = V(precomputed_vertex_out_weight_sums);                                     \
  a.init_v         = V(initial_guess_vertices);                                                 \
  a.init_val       = V(initial_guess_values);                                                   \
  a.alpha          = alpha;                                                                     \
  a.epsilon        = epsilon;                                                                   \
  a.max_iterations = max_iterations;                                                            \
  a.expensive      = do_expensive_check == TRUE;

cugraph_error_code_t cugraph_pagerank(const cugraph_resource_handle_t* handle, cugraph_graph_t* graph,
                                      const cugraph_type_erased_device_array_view_t* precomputed_vertex_out_weight_vertices,
                                      const cugraph_type_erased_device_array_view_t* precomputed_vertex_out_weight_sums,
                                      const cugraph_type_erased_device_array_view_t* initial_guess_vertices,
                                      const cugraph_type_erased_device_array_view_t* initial_guess_values, double alpha,
                                      double epsilon, size_t max_iterations, bool_t do_expensive_check,
                                      cugraph_centrality_result_t** result, cugraph_error_t** error)
{
  PR_ARGS_COMMON
  return pagerank_entry(handle, graph, a, true, result, error);
}

cugraph_error_code_t cugraph_pagerank_allow_nonconvergence(
  const cugraph_resource_handle_t* handle, cugraph_graph_t* graph,
  const cugraph_type_erased_device_array_view_t* precomputed_vertex_out_weight_vertices,
  const cugraph_type_erased_device_array_view_t* precomputed_vertex_out_weight_sums,
  const cugraph_type_erased_device_array_view_t* initial_guess_vertices,
  const cugraph_type_erased_device_array_view_t* initial_guess_values, double alpha, double epsilon,
  size_t max_iterations, bool_t do_expensive_check, cugraph_centrality_result_t** result, cugraph_error_t** error)
{
  PR_ARGS_COMMON
  return pagerank_entry(handle, graph, a, false, result, error);
}

cugraph_error_code_t cugraph_personalized_pagerank(
  const cugraph_resource_handle_t* handle, cugraph_graph_t* graph,
  const cugraph_type_erased_device_array_view_t* precomputed_vertex_out_weight_vertices,
  const cugraph_type_erased_device_array_view_t* precomputed_vertex_out_weight_sums,
  const cugraph_type_erased_device_array_view_t* initial_guess_vertices,
  const cugraph_type_erased_device_array_view_t* initial_guess_values,
  const cugraph_type_erased_device_array_view_t* personalization_vertices,
  const cugraph_type_erased_device_array_view_t* personalization_values, double alpha, double epsilon,
  size_t max_iterations, bool_t do_expensive_check, cugraph_centrality_result_t** result, cugraph_error_t** error)
{
  PR_ARGS_COMMON
  a.pers_v   = V(personalization_vertices);
  a.pers_val = V(personalization_values);
  return pagerank_entry(handle, graph, a, true, result, error);
}

cugraph_error_code_t cugraph_personalized_pagerank_allow_nonconvergence(
  const cugraph_resource_handle_t* handle, cugraph_graph_t* graph,
  const cugraph_type_erased_device_array_view_t* precomputed_vertex_out_weight_vertices,
  const cugraph_type_erased_device_array_view_t* precomputed_vertex_out_weight_sums,
  const cugraph_type_erased_device_array_view_t* initial_guess_vertices,
  const cugraph_type_erased_device_array_view_t* initial_guess_values,
  const cugraph_type_erased_device_array_view_t* personalization_vertices,
  const cugraph_type_erased_device_array_view_t* personalization_values, double alpha, double epsilon,
  size_t max_iterations, bool_t do_expensive_check, cugraph_centrality_result_t** result, cugraph_error_t** error)
{
  PR_ARGS_COMMON
  a.pers_v   = V(personalization_vertices);
  a.pers_val = V(personalization_values);
  return pagerank_entry(handle, graph, a, false, result, error);
}

// ------------------------------------------------------------------------ b200_ext.h bench hook
cugraph_error_code_t cugraph_b200_time_pull_spmv(const cugraph_resource_handle_t* handle, cugraph_graph_t* graph,
                                                 size_t iterations, double* ms_per_sweep,
                                                 double* algorithmic_bytes_per_sweep, cugraph_error_t** error)
{
  return guarded(error, [&] {
    auto const& h = H(handle);
    auto* g       = G(graph);
    B200_EXPECTS(g->mg == nullptr, CUGRAPH_NOT_IMPLEMENTED, "time_pull_spmv is single-GPU only");
    B200_EXPECTS(g->weight_type == FLOAT32, CUGRAPH_NOT_IMPLEMENTED, "time_pull_spmv: float32 graphs only");
    csx_t const& c = pull_view(h, *g);
    int32_t nv     = g->n_vertices;
    dbuf x = make_dbuf<float>(padded_x_elems(nv, sizeof(float)), h.stream), y = make_dbuf<float>(nv, h.stream);
    CUDA_TRY(cudaMemsetAsync(x.data(), 0, padded_x_elems(nv, sizeof(float)) * sizeof(float), h.stream));
    B200_LAUNCH(h, (k_fill<float>), grid_for(nv), kBlock, 0, x.as<float>(), nv, 1.0f / (float)nv);
    dbuf acc = make_dbuf<double>(acc_rows(c), h.stream);
    CUDA_TRY(cudaMemsetAsync(acc.data(), 0, sizeof(double) * acc_rows(c), h.stream));
    dbuf state = make_dbuf<pr_state_t>(1, h.stream);
    CUDA_TRY(cudaMemsetAsync(state.data(), 0, sizeof(pr_state_t), h.stream));
    auto sweep = [&] {
      if (c.offs64) launch_pull_sweep<int64_t, float>(h, c, x.as<float>(), y.as<float>(), acc.as<double>(), 0.85, state.as<pr_state_t>());
      else launch_pull_sweep_auto<int32_t, float>(h, c, nv, x.as<float>(), y.as<float>(), acc.as<double>(), 0.85, state.as<pr_state_t>());
    };
    for (int k = 0; k < 3; ++k) sweep();
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    CUDA_TRY(cudaEventRecord(e0, h.stream));
    for (size_t k = 0; k < iterations; ++k) sweep();
    CUDA_TRY(cudaEventRecord(e1, h.stream));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    check_last("time_pull_spmv");
    if (ms_per_sweep) *ms_per_sweep = (double)ms / (double)std::max<size_t>(iterations, 1);
    // SURVEY §8d: E*4 [indices] (+E*4 weights) + (V+1)*sizeof(offset) + V*4 [x] + V*4 [y]
    if (algorithmic_bytes_per_sweep)
      *algorithmic_bytes_per_sweep = (double)c.nnz * 4.0 * (g->weighted ? 2.0 : 1.0) +
                                     (double)(nv + 1) * (c.offs64 ? 8.0 : 4.0) + (double)nv * 8.0;
  });
}

// Debug hook: y of the sweep PageRank would use on this graph (the shared-memory piece stream when the graph has one)
// against the plain sweep (k_spmv_hi + k_spmv_low, an independent implementation) on the same pseudo-random x.  out[0..3] = degree >= 32 rows:
// max relative difference, its row, that row's degree, rows above 1e-5; out[4..7] = the same for the degree < 32 rows.
cugraph_error_code_t cugraph_b200_debug_compare_sweeps(const cugraph_resource_handle_t* handle, cugraph_graph_t* graph,
                                                       double* out, cugraph_error_t** error)
{
  return guarded(error, [&] {
    auto const& h = H(handle);
    auto* g       = G(graph);
    B200_EXPECTS(out != nullptr, CUGRAPH_INVALID_INPUT, "out is NULL");
    B200_EXPECTS(g->mg == nullptr && g->weight_type == FLOAT32, CUGRAPH_NOT_IMPLEMENTED, "single-GPU float32 graphs only");
    csx_t const& c = pull_view(h, *g);
    B200_EXPECTS(!c.offs64, CUGRAPH_NOT_IMPLEMENTED, "32-bit offsets only");
    const int32_t nv = g->n_vertices;
    const size_t px  = padded_x_elems(nv, sizeof(float));
    dbuf x = make_dbuf<float>(px, h.stream), y0 = make_dbuf<float>(nv, h.stream), y1 = make_dbuf<float>(nv, h.stream);
    CUDA_TRY(cudaMemsetAsync(x.data(), 0, px * sizeof(float), h.stream));
    B200_LAUNCH(h, (k_fill_pattern<float>), grid_for(nv), kBlock, 0, x.as<float>(), nv);
    dbuf acc = make_dbuf<double>(acc_rows(c), h.stream);
    CUDA_TRY(cudaMemsetAsync(acc.data(), 0, sizeof(double) * acc_rows(c), h.stream));
    dbuf state = make_dbuf<pr_state_t>(1, h.stream);
    CUDA_TRY(cudaMemsetAsync(state.data(), 0, sizeof(pr_state_t), h.stream));
    launch_pull_sweep<int32_t, float>(h, c, x.as<float>(), y0.as<float>(), acc.as<double>(), 0.85, state.as<pr_state_t>());
    launch_pull_sweep_auto<int32_t, float>(h, c, nv, x.as<float>(), y1.as<float>(), acc.as<double>(), 0.85, state.as<pr_state_t>());
    dbuf res = make_dbuf<unsigned long long>(4, h.stream);
    CUDA_TRY(cudaMemsetAsync(res.data(), 0, 4 * sizeof(unsigned long long), h.stream));
    B200_LAUNCH(h, (k_compare_rows<int32_t, float>), grid_for(c.n_rows), kBlock, 0, c.offsets.as<int32_t>(),
                c.row_vertex.as<int32_t>(), y0.as<float>(), y1.as<float>(), c.n_rows, c.seg[0], 1e-5,
                res.as<unsigned long long>(), res.as<unsigned long long>() + 2);
    unsigned long long hres[4];
    CUDA_TRY(cudaMemcpyAsync(hres, res.data(), sizeof(hres), cudaMemcpyDeviceToHost, h.stream));
    sync(h);
    for (int k = 0; k < 2; ++k) {
      const unsigned bits = (unsigned)(hres[k] >> 32);
      float rel;
      std::memcpy(&rel, &bits, sizeof(rel));
      const int32_t row = (int32_t)(hres[k] & 0xffffffffu);
      int32_t offs[2]   = {0, 0};
      if (c.n_rows > 0)
        CUDA_TRY(cudaMemcpy(offs, c.offsets.as<int32_t>() + row, sizeof(offs), cudaMemcpyDeviceToHost));
      out[4 * k + 0] = rel;
      out[4 * k + 1] = row;
      out[4 * k + 2] = offs[1] - offs[0];
      out[4 * k + 3] = (double)hres[2 + k];
    }
    check_last("debug_compare_sweeps");
  });
}

}  // extern "C"
