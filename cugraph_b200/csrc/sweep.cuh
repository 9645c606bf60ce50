// The shared-memory pull sweep: y[v] = init + alpha * sum_{(u->v)} x[u] * w(u,v) for EVERY row, gathers served from
// shared memory — per_v_transform_reduce_incoming_e specialised to reduce_op::plus and PageRank's e_op (reference
// cpp/include/cugraph/prims/detail/per_v_transform_reduce_e.cuh:389-885, cpp/src/link_analysis/pagerank_impl.cuh:262-287).
//
// Why: the plain sweep (spmv.cuh) is bound by the L2 -> SM path: every gather of x[src] costs a 32-byte L2 sector for
// 4 useful bytes (ncu r01: 0.86 L2 sectors per edge, lts 67 %, DRAM 16 %).  Here the source space is cut into blocks of W
// vertices whose x slice (192 KiB) a persistent CTA keeps in shared memory (TMA bulk copies + mbarrier), and the
// adjacency is re-laid as a stream of PIECES with 16-bit local column ids (sweep_layout_t, graph.cuh).
//
// Execution structure (round 2; ncu r02_ncu_x_md1: the round-1 kernel spent 58 % of its stall samples waiting on its
// id / row loads — one batch of loads in flight per warp, nothing while it processed them — and 7 % at CTA barriers):
//   * one 512-thread CTA per SM, 128 registers per thread.  A warp works on CHUNKS (a few step-rows of one kind, ~1-3 KiB of
//     ids + rows) and is double-buffered in REGISTERS: the 128-bit loads of chunk i+1 are issued before chunk i is
//     processed, its header before that, the draw of its index before that — no global-memory latency sits on the
//     critical path of a warp, and 16 warps x ~3 KiB are in flight per SM at all times (Little: 32 KiB needed).
//   * warps draw chunks from a per-phase cursor (one atomic per chunk, two draws ahead); there is no CTA barrier inside a
//     PHASE (= the chunks of one block in this CTA's range): barriers only where the slice changes.
//   * a CTA that finishes its own phases joins the phase with the most chunks left (same cursor: work stealing).
//   * a lane sums the 8 gathers of a slot as an fp32 tree and converts ONCE (the round-1 kernel issued one F2F + one DADD per
//     gather: 20 % of its instructions); slots, pieces and rows accumulate in fp64.
//   * one fp64 RED per piece into acc[row] (L2); the pieces of a hub row that fill a whole warp are summed by shuffles
//     first.  k_sweep_finish turns acc into y, clears it and resets the cursors.
#pragma once
#include "spmv.cuh"

namespace b200 {



constexpr int kSweepThreads = 512;  // 16 warps x 128 registers, two chunk buffers per warp (384 threads x 3 buffers: no faster)
constexpr int kSweepWarps   = kSweepThreads / 32;
constexpr int kSweepDynSmem = kHotSliceBytes;
constexpr int kTmaPiece     = 16 * 1024;  // bytes per bulk copy of the slice
constexpr int kStealMin     = 12;         // chunks a phase must have left for another CTA to load its slice and join

#ifndef B200_HOST_EMU
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity)
{
  asm volatile(
    "{\n"
    ".reg .pred p;\n"
    "WAIT_LOOP:\n"
    "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
    "@p bra DONE;\n"
    "bra WAIT_LOOP;\n"
    "DONE:\n"
    "}\n" ::"r"(smem_u32(bar)),
    "r"(parity)
    : "memory");
}
// TMA bulk copy global -> shared, completion signalled on the mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, uint64_t* bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                 smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ uint4 ld_stream_v4(const void* p)
{
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
// L2 eviction policies (createpolicy).  The 0.8 GB id / row stream is read once: marked evict-FIRST it leaves the L2 to the
// 59 MB of accumulators, whose REDs carry an evict-LAST policy (ncu r02: 57 % of the RED sectors missed the L2 and fetched
// their line from DRAM first).  RMAT-24: 0.331 -> 0.314 ms per sweep (profiles/r02_evict_ab*.log; a run-time choice per RED
// cost as much as the policy gains, so both are unconditional).
__device__ __forceinline__ unsigned long long make_l2_policy_evict_first()
{
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint4 ld_stream_v4(const void* p, unsigned long long pol)
{
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ uint2 ld_stream_v2(const void* p, unsigned long long pol)
{
  uint2 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.u32 {%0, %1}, [%2], %3;" : "=r"(v.x), "=r"(v.y) : "l"(p), "l"(pol));
  return v;
}
// fp64 accumulation with an L2 eviction policy on the accumulator line
__device__ __forceinline__ void red_acc(double* p, double v, unsigned long long acc_pol)
{
  asm volatile("red.global.add.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(p), "d"(v), "l"(acc_pol) : "memory");
}
__device__ __forceinline__ unsigned long long make_l2_policy_evict_last()
{
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ int ld_stream_i32(const int* p, unsigned long long pol)
{
  int v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ uint2 ld_stream_v2(const void* p)
{
  uint2 v;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
  return v;
}
__device__ __forceinline__ int ld_volatile(const int* p)
{
  int v;
  asm volatile("ld.volatile.global.s32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
#define B200_DYN_SMEM(name) extern __shared__ __align__(128) unsigned char name[]
#else  // host emulation (emu/cuda_runtime.h): a bulk copy is a memcpy by the issuing thread, waiting on the mbarrier is a
       // CTA barrier (every thread of the CTA waits on it in this kernel)
inline void mbar_init(uint64_t*, unsigned) {}
inline void mbar_expect_tx(uint64_t*, unsigned) {}
inline void mbar_wait(uint64_t*, unsigned) { __syncthreads(); }
inline void tma_bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, uint64_t*) { std::memcpy(dst_smem, src_gmem, bytes); }
inline uint4 ld_stream_v4(const void* p)
{
  uint4 v;
  std::memcpy(&v, p, sizeof(v));
  return v;
}
inline uint2 ld_stream_v2(const void* p)
{
  uint2 v;
  std::memcpy(&v, p, sizeof(v));
  return v;
}
inline int ld_volatile(const int* p) { return *p; }
inline unsigned long long make_l2_policy_evict_first() { return 0ull; }
inline uint4 ld_stream_v4(const void* p, unsigned long long) { return ld_stream_v4(p); }
inline uint2 ld_stream_v2(const void* p, unsigned long long) { return ld_stream_v2(p); }
inline int ld_stream_i32(const int* p, unsigned long long) { return *p; }
inline void red_acc(double* p, double v, unsigned long long) { *p += v; }
inline unsigned long long make_l2_policy_evict_last() { return 0ull; }
#define B200_DYN_SMEM(name) extern unsigned char name[] /* one CTA at a time: emu/emu_debug.cpp defines b200::smem_raw */
#endif

// ------------------------------------------------------------------------------------------
// per-lane arithmetic
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned lo16(unsigned v) { return v & 0xffffu; }
__device__ __forceinline__ unsigned hi16(unsigned v) { return v >> 16; }
__device__ __forceinline__ unsigned comp(uint4 const& v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w)); }

// the two entries packed in one 32-bit word of ids (weights wp[0], wp[1])
template <typename T, bool WEIGHTED>
__device__ __forceinline__ T pair_sum(unsigned ids, T const* __restrict__ sx, T const* wp)
{
  T a = sx[lo16(ids)], b = sx[hi16(ids)];
  if (WEIGHTED) {
    a *= wp[0];
    b *= wp[1];
  }
  return a + b;
}
// the 8 entries of a lane slot: summed as a tree in T (float: fp32 adds, ONE conversion), returned in fp64
template <typename T, bool WEIGHTED>
__device__ __forceinline__ double slot_sum(uint4 const& ids, T const* __restrict__ sx, T const* wp)
{
  const T a = pair_sum<T, WEIGHTED>(ids.x, sx, wp), b = pair_sum<T, WEIGHTED>(ids.y, sx, wp + 2);
  const T c = pair_sum<T, WEIGHTED>(ids.z, sx, wp + 4), d = pair_sum<T, WEIGHTED>(ids.w, sx, wp + 6);
  return (double)((a + b) + (c + d));
}

template <typename T>
__device__ __forceinline__ void load_w8(T (&wv)[8], T const* __restrict__ w, size_t slot)
{
#pragma unroll
  for (int k = 0; k < 8; ++k) wv[k] = ld_stream(w + slot * 8 + k);
}

// end of an F8 group (full 64-entry pieces): consecutive lanes may hold pieces of the same (hub) row — suffix-sum inside
// the runs first, run heads emit
__device__ __forceinline__ void emit_runs(double acc, int row, double* __restrict__ acc_out, int lane, unsigned long long acc_pol)
{
  const int r0 = __shfl_sync(0xffffffffu, row, 0);
  if (__all_sync(0xffffffffu, row == r0)) {  // 32 pieces of one hub row
    acc = warp_sum(acc);
    if (lane == 0 && r0 >= 0) red_acc(acc_out + r0, acc, acc_pol);
    return;
  }
  const int left = __shfl_up_sync(0xffffffffu, row, 1);
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const double nb = __shfl_down_sync(0xffffffffu, acc, o);
    const int rn    = __shfl_down_sync(0xffffffffu, row, o);
    if (lane + o < 32 && rn == row) acc += nb;
  }
  if (lane > 0 && left == row) row = -1;  // not the head of its run
  if (row >= 0) red_acc(acc_out + row, acc, acc_pol);
}

// ------------------------------------------------------------------------------------------
// a chunk in registers: up to 8 x 128 bits of ids / rows + 2 row words; what sits where depends on the kind
//   S  x 2 groups : q[3g] ids, q[3g+1], q[3g+2] the 8 rows
//   Q  x 4 groups : q[2g] ids, q[2g+1] the 4 rows
//   H  x 4 groups : q[g] ids, rows of groups (0,1) in q[4], of (2,3) in q[5]
//   F1 x 6 groups : q[g] ids, rows in q[6], q[7]
//   F2 x 3, F3 x 2: q[g*C+j] ids, rows in q[6]
//   F4 x 2        : q[g*4+j] ids, rows r0, r1
//   F5..F8 x 1    : q[j] ids, row r0
// ------------------------------------------------------------------------------------------
struct chunk_regs_t {
  uint4 q[8];
  int r0, r1;
};

struct sweep_ptrs_t {
  uint4 const* __restrict__ ids;
  int32_t const* __restrict__ rows;
  void const* __restrict__ w;
  double* __restrict__ acc;
  unsigned long long pol;      // L2 eviction policy of the stream loads
  unsigned long long acc_pol;  // of the accumulator REDs
};

template <int C, int G>
__device__ __forceinline__ void load_F(chunk_regs_t& b, sweep_chunk_t const& ch, sweep_ptrs_t const& p, int lane)
{
  uint4 const* ip   = p.ids + ((size_t)(unsigned)ch.sr_begin << 5) + lane;
  int32_t const* rp = p.rows + (size_t)(unsigned)ch.row_begin + lane;
#pragma unroll
  for (int g = 0; g < G; ++g) {
    if (g < ch.n_groups) {
#pragma unroll
      for (int j = 0; j < C; ++j) b.q[g * C + j] = ld_stream_v4(ip + ((g * C + j) << 5), p.pol);
      const int r = ld_stream_i32(rp + (g << 5), p.pol);
      if (C >= 4) {
        if (g == 0) b.r0 = r; else b.r1 = r;
      } else if (C == 1) {
        if (g == 0) b.q[6].x = r; else if (g == 1) b.q[6].y = r; else if (g == 2) b.q[6].z = r; else if (g == 3) b.q[6].w = r;
        else if (g == 4) b.q[7].x = r; else b.q[7].y = r;
      } else {
        if (g == 0) b.q[6].x = r; else if (g == 1) b.q[6].y = r; else b.q[6].z = r;
      }
    }
  }
}

template <typename T, bool WEIGHTED, int C, int G>
__device__ __forceinline__ void process_F(chunk_regs_t const& b, sweep_chunk_t const& ch, sweep_ptrs_t const& p,
                                          T const* __restrict__ sx, int lane)
{
#pragma unroll
  for (int g = 0; g < G; ++g) {
    if (g < ch.n_groups) {
      double s = 0.0;
#pragma unroll
      for (int j = 0; j < C; ++j) {
        T wv[8];
        if (WEIGHTED) load_w8<T>(wv, (T const*)p.w, ((size_t)(unsigned)(ch.sr_begin + g * C + j) << 5) + lane);
        s += slot_sum<T, WEIGHTED>(b.q[g * C + j], sx, wv);
      }
      int row;
      if (C >= 4) row = g == 0 ? b.r0 : b.r1;
      else if (C == 1) row = (int)(g < 4 ? comp(b.q[6], g) : comp(b.q[7], g - 4));
      else row = (int)comp(b.q[6], g);
      if (C == 8) emit_runs(s, row, p.acc, lane, p.acc_pol);
      else if (row >= 0) red_acc(p.acc + row, s, p.acc_pol);
    }
  }
}

// narrow kinds: ROWS rows per lane and step-row (S: 8, Q: 4, H: 2), G groups (= step-rows) per chunk
template <int ROWS, int G>
__device__ __forceinline__ void load_N(chunk_regs_t& b, sweep_chunk_t const& ch, sweep_ptrs_t const& p, int lane)
{
  uint4 const* ip   = p.ids + ((size_t)(unsigned)ch.sr_begin << 5) + lane;
  int32_t const* rp = p.rows + (size_t)(unsigned)ch.row_begin + (size_t)lane * ROWS;
#pragma unroll
  for (int g = 0; g < G; ++g) {
    if (g < ch.n_groups) {
      const uint4 ids = ld_stream_v4(ip + (g << 5), p.pol);
      if (ROWS == 8) {
        b.q[3 * g]     = ids;
        b.q[3 * g + 1] = ld_stream_v4(rp + g * 256, p.pol);
        b.q[3 * g + 2] = ld_stream_v4(rp + g * 256 + 4, p.pol);
      } else if (ROWS == 4) {
        b.q[2 * g]     = ids;
        b.q[2 * g + 1] = ld_stream_v4(rp + g * 128, p.pol);
      } else {
        b.q[g]        = ids;
        const uint2 r = ld_stream_v2(rp + g * 64, p.pol);
        uint4& dst    = b.q[4 + (g >> 1)];
        if (g & 1) {
          dst.z = r.x;
          dst.w = r.y;
        } else {
          dst.x = r.x;
          dst.y = r.y;
        }
      }
    }
  }
}

template <typename T, bool WEIGHTED, int ROWS, int G>
__device__ __forceinline__ void process_N(chunk_regs_t const& b, sweep_chunk_t const& ch, sweep_ptrs_t const& p,
                                          T const* __restrict__ sx, int lane)
{
#pragma unroll
  for (int g = 0; g < G; ++g) {
    if (g < ch.n_groups) {
      T wv[8];
      if (WEIGHTED) load_w8<T>(wv, (T const*)p.w, ((size_t)(unsigned)(ch.sr_begin + g) << 5) + lane);
      if (ROWS == 8) {
        const uint4 ids = b.q[3 * g];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const unsigned word = comp(ids, k >> 1);
          T v                 = sx[(k & 1) ? hi16(word) : lo16(word)];
          if (WEIGHTED) v *= wv[k];
          const int row = (int)comp(b.q[3 * g + 1 + (k >> 2)], k & 3);
          if (row >= 0) red_acc(p.acc + row, (double)v, p.acc_pol);
        }
      } else if (ROWS == 4) {
        const uint4 ids = b.q[2 * g];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const T v     = pair_sum<T, WEIGHTED>(comp(ids, k), sx, wv + 2 * k);
          const int row = (int)comp(b.q[2 * g + 1], k);
          if (row >= 0) red_acc(p.acc + row, (double)v, p.acc_pol);
        }
      } else {
        const uint4 ids = b.q[g];
        const uint4 rr  = b.q[4 + (g >> 1)];
        const T v0      = pair_sum<T, WEIGHTED>(ids.x, sx, wv) + pair_sum<T, WEIGHTED>(ids.y, sx, wv + 2);
        const T v1      = pair_sum<T, WEIGHTED>(ids.z, sx, wv + 4) + pair_sum<T, WEIGHTED>(ids.w, sx, wv + 6);
        const int row0 = (int)((g & 1) ? rr.z : rr.x), row1 = (int)((g & 1) ? rr.w : rr.y);
        if (row0 >= 0) red_acc(p.acc + row0, (double)v0, p.acc_pol);
        if (row1 >= 0) red_acc(p.acc + row1, (double)v1, p.acc_pol);
      }
    }
  }
}

// issue every load of the chunk (nothing is waited for); kind < 0: nothing to load
__device__ __forceinline__ void chunk_load(chunk_regs_t& b, sweep_chunk_t const& ch, sweep_ptrs_t const& p, int lane)
{
  switch (ch.kind) {
    case kKindS: load_N<8, 2>(b, ch, p, lane); break;
    case kKindQ: load_N<4, 4>(b, ch, p, lane); break;
    case kKindH: load_N<2, 4>(b, ch, p, lane); break;
    case kKindF1: load_F<1, 6>(b, ch, p, lane); break;
    case kKindF1 + 1: load_F<2, 3>(b, ch, p, lane); break;
    case kKindF1 + 2: load_F<3, 2>(b, ch, p, lane); break;
    case kKindF1 + 3: load_F<4, 2>(b, ch, p, lane); break;
    case kKindF1 + 4: load_F<5, 1>(b, ch, p, lane); break;
    case kKindF1 + 5: load_F<6, 1>(b, ch, p, lane); break;
    case kKindF1 + 6: load_F<7, 1>(b, ch, p, lane); break;
    case kKindF1 + 7: load_F<8, 1>(b, ch, p, lane); break;
    default: break;
  }
}

template <typename T, bool WEIGHTED>
__device__ __forceinline__ void chunk_process(chunk_regs_t const& b, sweep_chunk_t const& ch, sweep_ptrs_t const& p,
                                              T const* __restrict__ sx, int lane)
{
  switch (ch.kind) {
    case kKindS: process_N<T, WEIGHTED, 8, 2>(b, ch, p, sx, lane); break;
    case kKindQ: process_N<T, WEIGHTED, 4, 4>(b, ch, p, sx, lane); break;
    case kKindH: process_N<T, WEIGHTED, 2, 4>(b, ch, p, sx, lane); break;
    case kKindF1: process_F<T, WEIGHTED, 1, 6>(b, ch, p, sx, lane); break;
    case kKindF1 + 1: process_F<T, WEIGHTED, 2, 3>(b, ch, p, sx, lane); break;
    case kKindF1 + 2: process_F<T, WEIGHTED, 3, 2>(b, ch, p, sx, lane); break;
    case kKindF1 + 3: process_F<T, WEIGHTED, 4, 2>(b, ch, p, sx, lane); break;
    case kKindF1 + 4: process_F<T, WEIGHTED, 5, 1>(b, ch, p, sx, lane); break;
    case kKindF1 + 5: process_F<T, WEIGHTED, 6, 1>(b, ch, p, sx, lane); break;
    case kKindF1 + 6: process_F<T, WEIGHTED, 7, 1>(b, ch, p, sx, lane); break;
    case kKindF1 + 7: process_F<T, WEIGHTED, 8, 1>(b, ch, p, sx, lane); break;
    default: break;
  }
}

// ------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------
template <typename T>
struct sweep_args_t {
  sweep_ptrs_t p;
  sweep_chunk_t const* __restrict__ chunks;
  sweep_phase_t const* __restrict__ phases;
  int32_t const* __restrict__ cta_phase;
  int* __restrict__ cursor;
  T const* __restrict__ x;
  pr_state_t const* __restrict__ st;
  int n_phases;
  int W;
};

// ---- chunk supply of a warp.  Chunks are drawn from the phase's cursor in BATCHES of consecutive chunks (lane j holds
// the header of chunk base + j, one coalesced load), sized by what is left (remaining / 64, 1..8: long streams first,
// single chunks at the end of a phase so that the warps finish together).  The chain draw -> headers -> ids is three
// dependent round trips through L2 / HBM (~3 us); the draw of batch b+2 and the headers of batch b+1 are in flight while
// batch b is processed, the ids of chunk i+1 while chunk i is (ncu r02_ncu_sweep_v1/v2: with one chunk per stage a warp
// spent 4.5 us per chunk, 60 % of all stall samples on these three waits).
constexpr int kDrawMax = 8;

__device__ __forceinline__ int draw_want(int n, int seen)
{
  const int w = (n - seen) >> 6;
  return w < 1 ? 1 : (w > kDrawMax ? kDrawMax : w);
}
// lane 0 draws; the value is broadcast (draw_get) only when it is needed, a batch later
__device__ __forceinline__ int draw_issue(int* cursor, int want, int lane, bool more)
{
  int k = 0x3fffffff;
  if (more && lane == 0) k = atomicAdd(cursor, want);
  return k;
}
__device__ __forceinline__ int draw_get(int raw) { return __shfl_sync(0xffffffffu, raw, 0); }

__device__ __forceinline__ uint4 batch_headers(sweep_chunk_t const* __restrict__ chunks, int first, int cnt, int lane)
{
  uint4 v = make_uint4(0u, 0u, 0u, 0xffffffffu);  // kind = -1
  if (lane < cnt) v = ld_stream_v4(chunks + first + lane);
  return v;
}

// The headers of the current batch sit in a per-warp shared-memory ring (read back with one broadcast LDS per chunk);
// the headers of the next batch are a load in flight into `pend`, which is only touched at the next batch switch (kept in
// registers and copied with moves, ptxas hoisted the moves above the switch branch and every chunk waited for the load).
struct chunk_supply_t {
  sweep_chunk_t const* __restrict__ chunks;  // of the phase
  int* cursor;
  uint4* ring;  // [2][kDrawMax] of this warp
  int n;        // chunks in the phase
  uint4 pend;
  int cnt_cur, cnt_nxt, j, slot;
  int raw_nn, want_nn;  // draw in flight for the batch after `pend`

  __device__ __forceinline__ void start(sweep_chunk_t const* __restrict__ c, int* cur, uint4* warp_ring, int n_chunks, int lane)
  {
    chunks = c;
    cursor = cur;
    ring   = warp_ring;
    n      = n_chunks;
    const int w0 = draw_want(n, 0);
    const int r0 = draw_issue(cursor, w0, lane, true), r1 = draw_issue(cursor, w0, lane, true);
    const int b0 = draw_get(r0);
    cnt_cur      = b0 < n ? (n - b0 < w0 ? n - b0 : w0) : 0;
    const uint4 v0 = batch_headers(chunks, b0, cnt_cur, lane);
    const int b1 = draw_get(r1);
    cnt_nxt      = b1 < n ? (n - b1 < w0 ? n - b1 : w0) : 0;
    pend         = batch_headers(chunks, b1, cnt_nxt, lane);
    want_nn      = draw_want(n, b1 < n ? b1 + w0 : n);
    raw_nn       = draw_issue(cursor, want_nn, lane, b1 + w0 < n);
    j            = 0;
    slot         = 0;
    __syncwarp();  // the previous phase's readers of the ring are done
    if (lane < kDrawMax) ring[lane] = v0;
    __syncwarp();
  }
  __device__ __forceinline__ sweep_chunk_t next(int lane)
  {
    if (j == cnt_cur && cnt_cur > 0) {  // warp-uniform: the batch is used up
      slot ^= 1;
      if (lane < kDrawMax) ring[slot * kDrawMax + lane] = pend;  // its load was issued a batch ago
      __syncwarp();
      cnt_cur = cnt_nxt;
      j       = 0;
      const int b2 = draw_get(raw_nn);
      cnt_nxt      = b2 < n ? (n - b2 < want_nn ? n - b2 : want_nn) : 0;
      pend         = batch_headers(chunks, b2, cnt_nxt, lane);
      const int w3 = draw_want(n, b2 < n ? b2 + want_nn : n);
      raw_nn       = draw_issue(cursor, w3, lane, b2 + want_nn < n);
      want_nn      = w3;
    }
    sweep_chunk_t ch;
    ch.kind = -1;
    ch.n_groups = ch.sr_begin = ch.row_begin = 0;
    if (cnt_cur > 0) {
      const uint4 h = ring[slot * kDrawMax + j];
      ++j;
      ch.sr_begin  = (int)h.x;
      ch.row_begin = (int)h.y;
      ch.n_groups  = (int)h.z;
      ch.kind      = (int)h.w;
    }
    return ch;
  }
};

template <typename T, bool WEIGHTED>
__global__ void __launch_bounds__(kSweepThreads, 1) k_sweep(sweep_args_t<T> a)
{
  B200_DYN_SMEM(smem_raw);
  T* sx = reinterpret_cast<T*>(smem_raw);
  __shared__ uint64_t bar;
  __shared__ int s_best;
  __shared__ uint4 s_ring[kSweepWarps][2 * kDrawMax];
  if (a.st->done) return;
  a.p.pol        = make_l2_policy_evict_first();
  a.p.acc_pol    = make_l2_policy_evict_last();
  const int lane = threadIdx.x & 31;
  const int me   = (int)blockIdx.x;
  if (threadIdx.x == 0) mbar_init(&bar, 1);
  if (threadIdx.x < kHotZeroPad) sx[a.W + threadIdx.x] = (T)0;  // the zero columns every slice ends with
  const int own_lo = a.cta_phase[me], own_hi = a.cta_phase[me + 1];
  int next_own    = own_lo;
  unsigned parity = 0;
  int cur_block   = -1;
  while (true) {
    // ---- which phase next: the own ones in order, then the phase of another CTA with the most chunks left
    int p = -1;
    if (next_own < own_hi) {
      p = next_own++;
    } else {
      if (threadIdx.x == 0) s_best = 0;
      __syncthreads();
      int best = 0;
      for (int q = (int)threadIdx.x; q < a.n_phases; q += kSweepThreads) {
        if (q >= own_lo && q < own_hi) continue;
        const sweep_phase_t ph = a.phases[q];
        const int left         = (ph.chunk_end - ph.chunk_begin) - ld_volatile(a.cursor + q);
        if (left >= kStealMin && left > best) best = left;
      }
      if (best > 0) atomicMax(&s_best, best);
      __syncthreads();
      const int win = s_best;
      __syncthreads();
      if (win > 0) {
        if (threadIdx.x == 0) s_best = a.n_phases;
        __syncthreads();
        for (int q = (int)threadIdx.x; q < a.n_phases; q += kSweepThreads) {
          if (q >= own_lo && q < own_hi) continue;
          const sweep_phase_t ph = a.phases[q];
          const int left         = (ph.chunk_end - ph.chunk_begin) - ld_volatile(a.cursor + q);
          if (left >= kStealMin && left * 2 >= win) atomicMin(&s_best, q);
        }
        __syncthreads();
        p = s_best < a.n_phases ? s_best : -1;
      }
    }
    __syncthreads();  // every warp is done with the previous phase's slice (and has read s_best)
    if (p < 0) break;
    const sweep_phase_t ph = a.phases[p];
    const int n            = ph.chunk_end - ph.chunk_begin;
    const bool fresh       = ph.block != cur_block;
    if (fresh) {
      if (threadIdx.x == 0) {
        const unsigned bytes = (unsigned)(a.W * sizeof(T));
        mbar_expect_tx(&bar, bytes);
        const unsigned char* src = reinterpret_cast<const unsigned char*>(a.x + (size_t)ph.block * a.W);
        for (unsigned o = 0; o < bytes; o += kTmaPiece)
          tma_bulk_g2s(smem_raw + o, src + o, (bytes - o) < (unsigned)kTmaPiece ? (bytes - o) : (unsigned)kTmaPiece, &bar);
      }
      cur_block = ph.block;
    }
    // ---- the phase: chunk i is processed while the loads of i+1, the header of i+2 and the draw of i+3 are in flight
    chunk_supply_t sup;
    sup.start(a.chunks + ph.chunk_begin, a.cursor + p, s_ring[threadIdx.x >> 5], n, lane);
    sweep_chunk_t hA = sup.next(lane);
    sweep_chunk_t hB = sup.next(lane);
    chunk_regs_t A, B;
    chunk_load(A, hA, a.p, lane);
    if (fresh) {
      mbar_wait(&bar, parity);
      parity ^= 1;
    }
    while (hA.kind >= 0) {
      chunk_load(B, hB, a.p, lane);  // loads of chunk i+1
      const sweep_chunk_t hC = sup.next(lane);
      chunk_process<T, WEIGHTED>(A, hA, a.p, sx, lane);
      if (hB.kind < 0) break;
      chunk_load(A, hC, a.p, lane);
      const sweep_chunk_t hD = sup.next(lane);
      chunk_process<T, WEIGHTED>(B, hB, a.p, sx, lane);
      hA = hC;
      hB = hD;
    }
  }
}

// y[row] = acc * alpha + init for every covered row, init for the empty rows behind them; clears the accumulators and the
// cursors.  A warp handles 256 consecutive rows in four steps of 64: every step is one 512-byte load + one 512-byte store of
// accumulators and one 256-byte store of y per warp (lane = two rows), all four loads issued before the first use.
// (Eight CONSECUTIVE rows per thread looked the same on paper and ran at 2.3 TB/s: every warp-wide 128-bit access then
// touched sixteen 128-byte lines for a quarter of their bytes.)
template <typename T, int kFinishSteps>
__global__ void __launch_bounds__(256)
k_sweep_finish(double* __restrict__ acc, int n_cov, int n_rows, T* __restrict__ y, int32_t const* __restrict__ row_vertex,
               double alpha, int* __restrict__ cursor, int n_phases, pr_state_t const* __restrict__ st)
{
  if (st->done) return;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n_phases) cursor[t] = 0;
  const int lane = threadIdx.x & 31;
  const int base = (t >> 5) * (64 * kFinishSteps) + 2 * lane;  // first of this lane's two rows in step 0
  if (base - 2 * lane >= n_rows) return;
  const double init = st->init;
  double2 q[kFinishSteps];
#pragma unroll
  for (int k = 0; k < kFinishSteps; ++k) {
    const int r = base + 64 * k;
    q[k]        = make_double2(0.0, 0.0);
    if (r + 1 < n_cov) q[k] = *reinterpret_cast<double2*>(acc + r);
    else if (r < n_cov) q[k].x = acc[r];
  }
#pragma unroll
  for (int k = 0; k < kFinishSteps; ++k) {
    const int r = base + 64 * k;
    if (r + 1 < n_cov) *reinterpret_cast<double2*>(acc + r) = make_double2(0.0, 0.0);
    else if (r < n_cov) acc[r] = 0.0;
    const T v0 = (T)(q[k].x * alpha + init), v1 = (T)(q[k].y * alpha + init);
    if (!row_vertex && r + 1 < n_rows && sizeof(T) == 4) {
      *reinterpret_cast<float2*>(y + r) = make_float2((float)v0, (float)v1);
    } else {
      if (r < n_rows) y[row_vertex ? row_vertex[r] : r] = v0;
      if (r + 1 < n_rows) y[row_vertex ? row_vertex[r + 1] : r + 1] = v1;
    }
  }
}

// k_sweep alone: acc[row] += the row's sum; the caller turns acc into its result and clears acc and the cursors.
// x must hold padded_x_elems() elements, zero behind n_vertices (slices are copied whole)
template <typename T>
void launch_sweep_pieces(handle_impl const& h, sweep_layout_t const& L, T const* x, double* acc, pr_state_t const* st,
                         bool use_weights = true)
{
  // the attribute is per device and cheap to set: no process-wide "done" flag (a second device would miss it)
  const bool weighted = use_weights && L.w.data() != nullptr;
  if (weighted) CUDA_TRY(cudaFuncSetAttribute(k_sweep<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSweepDynSmem));
  else CUDA_TRY(cudaFuncSetAttribute(k_sweep<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSweepDynSmem));
  sweep_args_t<T> a;
  a.p.ids     = L.ids.as<uint4>();
  a.p.rows    = L.rows.as<int32_t>();
  a.p.w       = L.w.data();
  a.p.acc     = acc;
  a.chunks    = L.chunks.as<sweep_chunk_t>();
  a.phases    = L.phases.as<sweep_phase_t>();
  a.cta_phase = L.cta_phase.as<int32_t>();
  a.cursor    = L.cursor.as<int>();
  a.x         = x;
  a.st        = st;
  a.n_phases  = L.n_phases;
  a.W         = L.W;
  a.p.pol     = 0;
  a.p.acc_pol = 0;
  if (weighted) B200_LAUNCH(h, (k_sweep<T, true>), L.n_cta, kSweepThreads, kSweepDynSmem, a);
  else B200_LAUNCH(h, (k_sweep<T, false>), L.n_cta, kSweepThreads, kSweepDynSmem, a);
}

// x must hold padded_x_elems() elements, zero behind n_vertices (slices are copied whole)
template <typename T>
void launch_sweep(handle_impl const& h, csx_t const& c, sweep_layout_t const& L, T const* x, T* y, double* acc, double alpha,
                  pr_state_t const* st, bool use_weights = true, bool covered_rows_only = false)
{
  launch_sweep_pieces<T>(h, L, x, acc, st, use_weights);
  // 8 steps of 64 rows per warp: 0.335 ms per sweep against 0.340 with 4 and 0.354 with 2 (profiles/r02_fullchunk_ab.log)
  constexpr int kFinishSteps = 8;
  // covered_rows_only: y of the rows without edges already holds their (unvarying) value — multi-GPU blocks, where more than
  // half of the row slots are empty and the unvarying term is 0 (mg.cu)
  const int32_t finish_rows = covered_rows_only ? L.n_cov : c.n_rows;
  const int n = std::max((finish_rows + 2 * kFinishSteps - 1) / (2 * kFinishSteps), L.n_phases);  // threads: 16 rows each
  B200_LAUNCH(h, (k_sweep_finish<T, kFinishSteps>), (n + 255) / 256, 256, 0, acc, L.n_cov, finish_rows, y, c.row_vertex.as<int32_t>(), alpha,
              L.cursor.as<int>(), L.n_phases, st);
}

// dispatch: the piece stream when it exists for this graph, else the plain edge-balanced sweep
template <typename O, typename T>
void launch_pull_sweep_auto(handle_impl const& h, csx_t const& c, int32_t n_vertices, T const* x, T* y, double* acc,
                            double alpha, pr_state_t const* st, bool use_weights = true, bool covered_rows_only = false)
{
  sweep_layout_t const* L = sweep_layout(h, c, n_vertices, sizeof(T));
  if (!L) launch_pull_sweep<O, T>(h, c, x, y, acc, alpha, st, use_weights);  // the plain sweep writes every row
  else launch_sweep<T>(h, c, *L, x, y, acc, alpha, st, use_weights, covered_rows_only);
}

// elements an x buffer needs: whole slices are TMA-copied and everything behind n_vertices must read 0.
// The buffer must be zero-filled once at allocation; only [0, n_vertices) is ever written afterwards.
inline size_t padded_x_elems(int32_t n_vertices, size_t elem_size)
{
  const size_t slice = kHotSliceBytes / elem_size;
  const size_t W     = slice - kHotZeroPad;
  return ((size_t)n_vertices / W + 2) * slice;
}

}  // namespace b200
