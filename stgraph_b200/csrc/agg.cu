// Fused neighbour aggregation (gather - scale - sum) for sm_100a.
//
//   out[r,:] = row_scale[r] * sum_{e in row r} nbr_scale[col[e]] * edge_scale[eid(e)] * x[col[e],:]
//
// This is the one kernel shape on STGraph's hot path: the reference emits it
// from stgraph/compiler/code_gen/templates/fa/tpl_fa_csr*.jinja:1-57 with one
// thread per (row, feature) and a serial edge loop of scalar loads.  Here:
//   * a GROUP of lanes (1..32, power of two) owns a row and each lane owns VEC
//     (1/2/4) consecutive floats x NACC chunks, so one neighbour row is fetched
//     with 128-bit coalesced loads;
//   * column indices / scales of the next GROUP edges are loaded cooperatively
//     (one coalesced load per group) and prefetched one batch ahead, then
//     broadcast with warp shuffles;
//   * UNROLL independent neighbour-row loads are in flight per lane;
//   * rows longer than hub_threshold go to a block-per-row kernel whose warps
//     split the row and reduce through shared memory in a fixed order
//     (deterministic: no atomics anywhere).
// Measured alternatives that LOST on B200 and were removed (profiles/r01_agg_ncu.md, sources kept in
// scripts/agg_variants_r01.cu.txt): a multi-row streaming variant (more instructions, fewer warps),
// a cp.async (LDGSTS) shared-memory ring and a cp.async.bulk (UBLKCP) ring: the gather is bound by the
// L2->SM fabric (~6-7.5 TB/s of gathered rows), not by the bytes in flight.
// Memory bound: HBM roofline; algorithmic bytes per launch
//   4*(2*N*F + E + (N+1) + 2*N [+ E for edge_scale]).
#include "common.cuh"

#include <cooperative_groups.h>

#include <algorithm>
#include <cstdlib>

namespace stg {
namespace {

constexpr int kBlockThreads = 256;
constexpr int kHubThreads = 512;

template <int VEC>
__device__ __forceinline__ typename VecT<VEC>::type ld_row(const float* p) {
  using T = typename VecT<VEC>::type;
  return __ldg(reinterpret_cast<const T*>(p));
}
template <int VEC>
__device__ __forceinline__ void st_row(float* p, typename VecT<VEC>::type v) {
  using T = typename VecT<VEC>::type;
  __stcs(reinterpret_cast<T*>(p), v);
}

struct AggParams {
  const int32_t* __restrict__ row_off;
  const int32_t* __restrict__ col;
  const int32_t* __restrict__ eids;
  const int32_t* __restrict__ hub_rows;
  const int32_t* __restrict__ hub_count;
  const int32_t* __restrict__ out_rows;   // view row -> output row (NULL: identity)
  const int2* __restrict__ meta;          // PACKED mode: {column, scale bits} of every CSR slot (stg_csr_pack_edge_meta_f32)
  int* queue;                             // global row queue {next chunk, finished blocks} (StgCsrView::work_queue) or NULL
  int num_rows;
  int num_edges;
  int eid_base;
  int eids_identity;
  int hub_threshold;
  int hub_capacity;
  const float* __restrict__ x;    // already offset to the chunk's first column
  float* __restrict__ out;        // same
  int ld;                         // floats between consecutive rows of x (>= feat)
  int ld_out;                     // floats between consecutive rows of out (>= feat)
  int width;                      // floats of this chunk handled by the launch
  const float* __restrict__ ns;
  const float* __restrict__ es;
  const float* __restrict__ rs;
  // Row-partitioned source matrix (multi-GPU): block q holds rows [bounds[q], bounds[q+1]) and may
  // live in a PEER GPU's memory (NVLink loads); nparts == 0 means one local matrix `x`.
  int accumulate;     // 0: out = result; 1: out += result (read-modify-write); 2: out += result with red.global.add
  int nparts;
  int bounds[STG_MAX_PARTS + 1];
  const float* xs[STG_MAX_PARTS];
};

// out += v with a vector reduction (red.global.add.v4.f32 on sm_90+): no read round trip
__device__ __forceinline__ void red_add(float* p, float v) { atomicAdd(p, v); }
__device__ __forceinline__ void red_add(float* p, float2 v) { atomicAdd(reinterpret_cast<float2*>(p), v); }
__device__ __forceinline__ void red_add(float* p, float4 v) { atomicAdd(reinterpret_cast<float4*>(p), v); }

// Address of source row c in the owner's block of a row-partitioned matrix.
__device__ __forceinline__ const float* src_row(const AggParams& p, int c) {
  int o = 0;
#pragma unroll
  for (int q = 1; q < STG_MAX_PARTS; ++q) o += (q < p.nparts && c >= p.bounds[q]) ? 1 : 0;
  return p.xs[o] + static_cast<size_t>(c - p.bounds[o]) * p.ld;
}

// How the edge loop finds a neighbour row and its scale:
//   kPlain   column_indices[e], then the dependent gathers nbr_scale[col] (* edge_scale[eid]);
//   kParts   as kPlain, source matrix row-partitioned over peer GPUs (cold path, stg_agg_scaled_sum_parts_f32);
//   kPacked  ONE coalesced 8-byte load per edge: {col, nbr_scale[col] * edge_scale[eid]} precomputed per CSR slot
//            (stg_csr_pack_edge_meta_f32).  The scattered 4-byte nbr_scale gather costs one 32-byte L2 sector
//            request per edge -- as many requests as a quarter of the 400..512-byte neighbour row itself -- and
//            one level of the dependent load chain; a static graph with a fixed norm pays for the packing once.
enum AggMode { kPlain = 0, kParts = 1, kPacked = 2 };

// Column index (and, kPacked, the scale `ms`) of edge `base + gl` (0 / 0.f past the end of the row).
template <int MODE>
__device__ __forceinline__ void load_col(const AggParams& p, int base, int end, int gl, int& c, float& ms) {
  c = 0;
  ms = 0.f;
  const int e = base + gl;
  if (e < end) {
    if constexpr (MODE == kPacked) {
      const int2 m = __ldcs(p.meta + e);
      c = m.x;
      ms = __int_as_float(m.y);
    } else {
      c = ld_stream(p.col + e);
    }
  }
}
// Combined scale of edge `base + gl` whose column `c` has arrived (0.f past the end of the row).
template <int MODE>
__device__ __forceinline__ void load_scale(const AggParams& p, int base, int end, int gl, int c, float ms, float& s) {
  if constexpr (MODE == kPacked) {
    s = ms;
    return;
  }
  s = 0.f;
  const int e = base + gl;
  if (e < end) {
    float sc = 1.f;
    if (p.ns) sc = __ldg(p.ns + c);
    if (p.es) {
      const int eid = p.eids_identity ? e : (ld_stream(p.eids + e) - p.eid_base);
      sc *= __ldg(p.es + eid);
    }
    s = sc;
  }
}

// Accumulate edges [beg,end) visited with stride `step` batches of GROUP edges,
// starting at batch `first`.  All lanes of a group execute this together.
// (my_c, my_s) = column / scale of the first batch, loaded by the caller (so that a caller can
// have them in flight long before the row is processed).
// Neighbour-row loads of one lane: a row address is ONE IMAD.WIDE off a per-lane base pointer; lanes past
// `width` are switched off by a loop-invariant predicate (their sums are never written).
template <int VEC, int GROUP, int NACC, int MODE>
struct RowLoader {
  using T = typename VecT<VEC>::type;
  const char* base[NACC];
  int off[NACC];
  bool live[NACC];        // lane-constant: this lane's chunk k lies inside the row
  unsigned ld_bytes;
  __device__ __forceinline__ RowLoader(const AggParams& p, int gl) {
    ld_bytes = static_cast<unsigned>(p.ld) * 4u;
#pragma unroll
    for (int k = 0; k < NACC; ++k) {
      int o = (gl + k * GROUP) * VEC;
      live[k] = o < p.width;
      if (!live[k]) o = (p.width - 1) / VEC * VEC;
      off[k] = o;
      base[k] = reinterpret_cast<const char*>(p.x + o);
    }
  }
  // Idle lanes (F=100: lanes 25..31) are predicated off with a loop-invariant predicate: a lane that does not
  // load costs no LSU write-back slot, and the write-back of 32 x 16 bytes per row is what bounds F = 68..124.
  __device__ __forceinline__ T load(const AggParams& p, int c, int k) const {
    T v;
    zero_vec(v);
    if constexpr (MODE == kParts) {
      v = ld_row<VEC>(src_row(p, c) + off[k]);
    } else {
      if (live[k]) v = __ldg(reinterpret_cast<const T*>(base[k] + static_cast<unsigned long long>(static_cast<unsigned>(c)) * ld_bytes));
    }
    return v;
  }
};

// Accumulate edges [beg,end) visited with stride `step` batches of GROUP edges,
// starting at batch `first`.  All lanes of a group execute this together.
// (my_c, my_s) = column / scale of the first batch, loaded by the caller (so that a caller can
// have them in flight long before the row is processed).
template <int VEC, int GROUP, int NACC, int UNROLL_ = 0, int MODE = kPlain>
__device__ __forceinline__ void accumulate_edges(const AggParams& p, int beg, int end, int first_batch,
                                                 int batch_step, int gl, unsigned gmask,
                                                 typename VecT<VEC>::type (&acc)[NACC], int my_c, float my_s) {
  using T = typename VecT<VEC>::type;
  constexpr int UNROLL = UNROLL_ > 0 ? (UNROLL_ < GROUP ? UNROLL_ : GROUP) : (GROUP >= 8 ? 8 : GROUP) / (NACC > 2 ? 2 : 1);
  const RowLoader<VEC, GROUP, NACC, MODE> rows(p, gl);

  // (column, scale) of the batch a lane group is summing reach the other lanes either by two SHFL per edge
  // or through shared memory (one STS.64 per lane + one LDS.128 per TWO edges).  A/B on one box, config 5:
  // sub-warp groups (F=64, GROUP=16) 2.04 ms through shared memory against 2.34 ms with shuffles; full-warp
  // groups (F=100 / 128) 2.92 / 3.07 ms against 2.79 / 2.82 ms -- so each geometry takes its winner.
  constexpr bool kSmemMeta = GROUP < 32;
  __shared__ int2 meta[kSmemMeta ? kHubThreads : 1];
  const int2* gmeta = meta + (threadIdx.x & ~(GROUP - 1));
  auto fetch_meta = [&](int j, int (&c)[UNROLL], float (&sc)[UNROLL]) {
    if constexpr (!kSmemMeta) {
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        c[u] = __shfl_sync(gmask, my_c, j + u, GROUP);
        sc[u] = __shfl_sync(gmask, my_s, j + u, GROUP);
      }
    } else if constexpr (UNROLL == 1) {
      c[0] = gmeta[j].x;
      sc[0] = __int_as_float(gmeta[j].y);
    } else {
#pragma unroll
      for (int u = 0; u < UNROLL; u += 2) {
        const int4 m = *reinterpret_cast<const int4*>(gmeta + j + u);
        c[u] = m.x;
        sc[u] = __int_as_float(m.y);
        c[u + 1] = m.z;
        sc[u + 1] = __int_as_float(m.w);
      }
    }
  };

  int base = beg + first_batch * GROUP;
  int nx_c;
  float nx_m, nx_s;
  for (; base < end; base += batch_step * GROUP) {
    if constexpr (kSmemMeta) {
      __syncwarp(gmask);                                     // the previous batch has been read by every lane
      meta[threadIdx.x] = make_int2(my_c, __float_as_int(my_s));
      __syncwarp(gmask);
    }
    load_col<MODE>(p, base + batch_step * GROUP, end, gl, nx_c, nx_m);   // prefetch next batch
    load_scale<MODE>(p, base + batch_step * GROUP, end, gl, nx_c, nx_m, nx_s);
    const int n = min(GROUP, end - base);
    int j = 0;
    for (; j + UNROLL <= n; j += UNROLL) {     // full groups: UNROLL unpredicated row loads in flight
      int c[UNROLL];
      float sc[UNROLL];
      T v[UNROLL][NACC];
      fetch_meta(j, c, sc);
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
#pragma unroll
        for (int k = 0; k < NACC; ++k) v[u][k] = rows.load(p, c[u], k);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
#pragma unroll
        for (int k = 0; k < NACC; ++k) fma_vec(acc[k], sc[u], v[u][k]);
      }
    }
    if (j < n) {                               // last, partial group of the batch
      int c[UNROLL];
      float sc[UNROLL];
      T v[UNROLL][NACC];
      fetch_meta(j, c, sc);
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
          if ((j + u) < n) v[u][k] = rows.load(p, c[u], k);
          else zero_vec(v[u][k]);
        }
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
#pragma unroll
        for (int k = 0; k < NACC; ++k) fma_vec(acc[k], sc[u], v[u][k]);
      }
    }
    my_c = nx_c;
    my_s = nx_s;
  }
}

template <int VEC, int GROUP, int NACC, int MODE = kPlain>
__device__ __forceinline__ void accumulate_edges(const AggParams& p, int beg, int end, int first_batch,
                                                 int batch_step, int gl, unsigned gmask,
                                                 typename VecT<VEC>::type (&acc)[NACC]) {
  int c;
  float m, s;
  load_col<MODE>(p, beg + first_batch * GROUP, end, gl, c, m);
  load_scale<MODE>(p, beg + first_batch * GROUP, end, gl, c, m, s);
  accumulate_edges<VEC, GROUP, NACC, 0, MODE>(p, beg, end, first_batch, batch_step, gl, gmask, acc, c, s);
}

template <typename T>
__device__ __forceinline__ T shfl_xor_vec(T v, int o);
template <>
__device__ __forceinline__ float shfl_xor_vec<float>(float v, int o) { return __shfl_xor_sync(0xffffffffu, v, o); }
template <>
__device__ __forceinline__ float2 shfl_xor_vec<float2>(float2 v, int o) {
  return make_float2(__shfl_xor_sync(0xffffffffu, v.x, o), __shfl_xor_sync(0xffffffffu, v.y, o));
}
template <>
__device__ __forceinline__ float4 shfl_xor_vec<float4>(float4 v, int o) {
  return make_float4(__shfl_xor_sync(0xffffffffu, v.x, o), __shfl_xor_sync(0xffffffffu, v.y, o),
                     __shfl_xor_sync(0xffffffffu, v.z, o), __shfl_xor_sync(0xffffffffu, v.w, o));
}


// PAIR form of the edge loop for one row per warp with 16 < F/4 <= 32 (F = 68..128): the two half-warps
// sum ALTERNATE edges of the row, each half covering the row with 16 lanes x 2 float4 chunks, so ONE
// SHFL.IDX pair (per-lane source: lane j + half) hands two edges their {column, scale}.  ncu on config 5,
// F=100 (profiles/r01_agg_ncu.md): the LSU data pipe is the busiest unit (77 % of peak), and the two
// 32-lane broadcasts per edge are a third of its wavefronts; the halves' partial sums are merged once per
// row with four SHFL.BFLY.  Fixed order: deterministic.  On return lane L holds the row's floats [4L, 4L+4).
// Neighbour-row load of the pair form: a plain read-only load.  Measured alternatives on config 5 (4.84 ms/step):
// L2 evict_last policy 4.80-4.85 ms (noise), no L1 allocation 6.24 ms (the 7 % of sectors that hit L1 matter).
__device__ __forceinline__ float4 ldg_row(const float4* p) { return __ldg(p); }

// (Measured and dropped, r2: per-edge L2 eviction hints -- ld.global.L2::cache_hint with an evict_first policy for
// sources further than a window of ids from the row, evict_last for the near ones, selected without a branch --
// 2.22-2.32 ms against 2.15 ms on config 5: the policy select costs more issue slots than the hit rate returns.)
template <int UNROLL, int MODE>
__device__ __forceinline__ void accumulate_edges_pair(const AggParams& p, int beg, int end, int lane, float4& result,
                                                      int my_c, float my_m, float my_s) {
  static_assert(UNROLL % 2 == 0, "two edges per step");
  constexpr int STEPS = UNROLL / 2;
  const int half = lane >> 4;
  const int hl = lane & 15;
  const unsigned ld_bytes = static_cast<unsigned>(p.ld) * 4u;
  const char* base0;
  const char* base1;
  {
    const int last = (p.width - 1) / 4 * 4;
    int o0 = hl * 4, o1 = (hl + 16) * 4;
    if (o0 > last) o0 = last;
    if (o1 > last) o1 = last;
    base0 = reinterpret_cast<const char*>(p.x + o0);
    base1 = reinterpret_cast<const char*>(p.x + o1);
  }
  const bool live1 = (hl + 16) * 4 < p.width;   // chunk 0 is always inside the row (width > 64); F=100: 9 of 16 lanes
  auto row0 = [&](int c) { return ldg_row(reinterpret_cast<const float4*>(base0 + static_cast<unsigned long long>(static_cast<unsigned>(c)) * ld_bytes)); };
  auto row1 = [&](int c) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (live1) v = ldg_row(reinterpret_cast<const float4*>(base1 + static_cast<unsigned long long>(static_cast<unsigned>(c)) * ld_bytes));
    return v;
  };
  float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0;
  (void)my_m;
  for (int base = beg; base < end; base += 32) {
    int nx_c;
    float nx_m, nx_s;
    load_col<MODE>(p, base + 32, end, lane, nx_c, nx_m);   // prefetch next batch
    load_scale<MODE>(p, base + 32, end, lane, nx_c, nx_m, nx_s);
    const int n = min(32, end - base);
    int j = 0;
    for (; j + UNROLL <= n; j += UNROLL) {     // full groups: UNROLL edges = STEPS unpredicated steps per half
      int c[STEPS];
      float sc[STEPS];
      float4 v0[STEPS], v1[STEPS];
#pragma unroll
      for (int u = 0; u < STEPS; ++u) {
        c[u] = __shfl_sync(0xffffffffu, my_c, j + 2 * u + half);
        sc[u] = __shfl_sync(0xffffffffu, my_s, j + 2 * u + half);
      }
#pragma unroll
      for (int u = 0; u < STEPS; ++u) {
        v0[u] = row0(c[u]);
        v1[u] = row1(c[u]);
      }
#pragma unroll
      for (int u = 0; u < STEPS; ++u) {
        fma_vec(acc0, sc[u], v0[u]);
        fma_vec(acc1, sc[u], v1[u]);
      }
    }
    if (j < n) {                               // last, partial group of the batch
      int c[STEPS];
      float sc[STEPS];
      float4 v0[STEPS], v1[STEPS];
#pragma unroll
      for (int u = 0; u < STEPS; ++u) {
        c[u] = __shfl_sync(0xffffffffu, my_c, (j + 2 * u + half) & 31);
        sc[u] = __shfl_sync(0xffffffffu, my_s, (j + 2 * u + half) & 31);
      }
#pragma unroll
      for (int u = 0; u < STEPS; ++u) {
        if ((j + 2 * u + half) < n) {
          v0[u] = row0(c[u]);
          v1[u] = row1(c[u]);
        } else {
          zero_vec(v0[u]);
          zero_vec(v1[u]);
          sc[u] = 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < STEPS; ++u) {
        fma_vec(acc0, sc[u], v0[u]);
        fma_vec(acc1, sc[u], v1[u]);
      }
    }
    my_c = nx_c;
    my_s = nx_s;
  }
  // merge the halves: lane L (half 0) owns chunk 0 = floats [4L, 4L+4), lane L (half 1) owns chunk 1 = [4L, 4L+4) too
  const float4 give = half ? acc0 : acc1;      // what the partner lane owns
  float4 mine = half ? acc1 : acc0;
  add_vec(mine, shfl_xor_vec<float4>(give, 16));
  result = mine;
}

// Scaled row result -> out (assign / += / red.add).
template <int VEC, int GROUP, int NACC>
__device__ __forceinline__ void write_row(const AggParams& p, int row, int gl, bool nonempty, float r,
                                          typename VecT<VEC>::type (&acc)[NACC], bool have_old,
                                          typename VecT<VEC>::type (&old)[NACC]) {
  using T = typename VecT<VEC>::type;
  float* dst = p.out + static_cast<size_t>(row) * p.ld_out;
#pragma unroll
  for (int k = 0; k < NACC; ++k) {
    const int o = (gl + k * GROUP) * VEC;
    if (o < p.width) {
      scale_vec(acc[k], r);
      if (p.accumulate == 2) {
        if (nonempty) red_add(dst + o, acc[k]);
        continue;
      }
      if (p.accumulate) add_vec(acc[k], have_old ? old[k] : *reinterpret_cast<const T*>(dst + o));
      st_row<VEC>(dst + o, acc[k]);
    }
  }
}

template <int VEC, int GROUP, int NACC>
__device__ __forceinline__ void write_row(const AggParams& p, int row, int gl, bool nonempty, float r,
                                          typename VecT<VEC>::type (&acc)[NACC]) {
  typename VecT<VEC>::type none[NACC];
#pragma unroll
  for (int k = 0; k < NACC; ++k) zero_vec(none[k]);
  write_row<VEC, GROUP, NACC>(p, row, gl, nonempty, r, acc, false, none);
}

// accumulate == 1 (out += ...): the row's current value, requested BEFORE its edges are walked so that the read
// overlaps the gathers (the halo-source pass of the multi-GPU path: ~2.5 edges per row, where a second dependent
// DRAM round trip per row doubled the pass).
template <int VEC, int GROUP, int NACC>
__device__ __forceinline__ void prefetch_row(const AggParams& p, int row, int gl, typename VecT<VEC>::type (&old)[NACC]) {
  using T = typename VecT<VEC>::type;
  const float* dst = p.out + static_cast<size_t>(row) * p.ld_out;
#pragma unroll
  for (int k = 0; k < NACC; ++k) {
    const int o = (gl + k * GROUP) * VEC;
    zero_vec(old[k]);
    if (o < p.width) old[k] = *reinterpret_cast<const T*>(dst + o);
  }
}

// Software-pipelined row queue.  A block owns `slots_per_block` consecutive row slots (a slot =
// 32/GROUP rows, one per lane group); its warps draw slots from a shared-memory counter, so a warp
// that got short rows simply takes more of them (one-row-per-warp blocks idle 1/3 of their warp slots
// on a power-law graph: every block waits for its longest row).  The dependent load chain of a row
// (row_offset -> column index -> neighbour scale -> neighbour rows) is spread over four consecutive
// loop iterations: while row i is being summed, the scales of row i+1, the columns of row i+2 and
// the offsets of row i+3 are already in flight.
//
// GQ (global queue) form: a persistent grid (resident blocks only) whose WARPS draw chunks of `slots_per_block`
// consecutive slots from ONE device-wide counter (StgCsrView::work_queue), the next chunk id being fetched while
// the current chunk is summed.  All resident warps then work inside one narrow, moving window of destination
// rows (4736 warps x 8 rows = 38 K rows, 15 MB of x on config 5, against the 151 K-row window of 592 resident
// 256-row blocks), so the source rows of a community graph are re-read from L2, not from HBM, and no block
// waits for its longest row at the tail.  The last block to finish resets the counters for the next launch.
template <int VEC, int GROUP, int NACC, int MINB, int UNROLL, int MODE, bool PAIR = false, bool GQ = false>
__global__ void __launch_bounds__(kBlockThreads, MINB) agg_rows_pipe_kernel(const AggParams p, int slots_per_block) {
  using T = typename VecT<VEC>::type;
  constexpr int GPW = 32 / GROUP;
  __shared__ int next_slot;
  const int lane = threadIdx.x & 31;
  const int gl = lane & (GROUP - 1);
  const int gidx = lane / GROUP;
  const unsigned gmask = (GROUP == 32) ? 0xffffffffu : (((1u << GROUP) - 1u) << (lane & ~(GROUP - 1)));
  const int total_slots = (p.num_rows + GPW - 1) / GPW;
  const int first = GQ ? 0 : blockIdx.x * slots_per_block;
  const int last = GQ ? total_slots : min(first + slots_per_block, total_slots);
  int q_cur = 0, q_pos = slots_per_block, q_nxt = 0;   // GQ: chunk being walked, position in it, chunk id in flight
  if constexpr (GQ) {
    if (lane == 0) q_nxt = atomicAdd(p.queue, 1);
  } else {
    if (threadIdx.x == 0) next_slot = first;
    __syncthreads();
  }

  auto draw = [&]() {
    if constexpr (GQ) {
      if (q_pos == slots_per_block && q_cur < total_slots) {      // warp-uniform
        q_cur = __shfl_sync(0xffffffffu, q_nxt, 0) * slots_per_block;
        q_pos = 0;
        if (lane == 0 && q_cur < total_slots) q_nxt = atomicAdd(p.queue, 1);
      }
      return q_cur + q_pos++;
    } else {
      int s = 0;
      if (lane == 0) s = atomicAdd(&next_slot, 1);
      return __shfl_sync(0xffffffffu, s, 0);
    }
  };
  auto finish = [&]() {
    if constexpr (GQ) {          // the last block to get here has seen every chunk drawn: rearm the queue
      __syncthreads();
      if (threadIdx.x == 0 && atomicAdd(p.queue + 1, 1) == static_cast<int>(gridDim.x) - 1) {
        p.queue[0] = 0;
        p.queue[1] = 0;
        __threadfence();
      }
    }
    grid_dependency_wait();
  };
  // stage A: slot -> output row, [beg, end); end = -1 when there is nothing to do (past the end, hub row)
  auto stage_a = [&](int slot, int& row, int& beg, int& end) {
    row = slot * GPW + gidx;
    if (slot >= last || row >= p.num_rows) { row = 0; beg = 0; end = -1; return; }
    beg = __ldg(p.row_off + row);
    end = __ldg(p.row_off + row + 1);
    if (p.out_rows) row = __ldg(p.out_rows + row);
  };
  auto drop_hub = [&](int& beg, int& end) {
    if (p.hub_threshold > 0 && (end - beg) > p.hub_threshold) beg = 0, end = -1;
  };

  int slot0, row0, beg0, end0, c0;     // row being summed (scale loaded at the top of the iteration)
  int row1, beg1, end1, c1;            // columns in flight
  int row2, beg2, end2;                // offsets in flight
  float s0, r0, m0, m1;                // m*: scale that arrived WITH the column (kPacked)
  slot0 = draw();
  if (slot0 >= last) { finish(); return; }
  stage_a(slot0, row0, beg0, end0);
  int slot1 = draw();
  stage_a(slot1, row1, beg1, end1);
  int slot2 = draw();
  stage_a(slot2, row2, beg2, end2);
  drop_hub(beg0, end0);
  load_col<MODE>(p, beg0, end0, gl, c0, m0);
  drop_hub(beg1, end1);
  load_col<MODE>(p, beg1, end1, gl, c1, m1);
  load_scale<MODE>(p, beg0, end0, gl, c0, m0, s0);
  r0 = (end0 >= 0 && p.rs) ? __ldg(p.rs + row0) : 1.f;

  while (slot0 < last) {
    // issue the loads of the three younger stages before touching the current row
    const int slot3 = draw();
    int row3, beg3, end3;
    stage_a(slot3, row3, beg3, end3);
    drop_hub(beg2, end2);
    int c2;
    float m2;
    load_col<MODE>(p, beg2, end2, gl, c2, m2);
    float s1;
    load_scale<MODE>(p, beg1, end1, gl, c1, m1, s1);
    const float r1 = (end1 >= 0 && p.rs) ? __ldg(p.rs + row1) : 1.f;

    if (end0 >= 0) {
      T acc[NACC];
      T old[NACC];
      const bool rmw = NACC <= 2 && p.accumulate == 1;       // wider tiles have no registers to spare for it
      if constexpr (NACC <= 2) {
        if (rmw) prefetch_row<VEC, GROUP, NACC>(p, row0, gl, old);
      }
      if constexpr (PAIR) {
        static_assert(VEC == 4 && GROUP == 32 && NACC == 1, "pair form: one row per warp, float4 lanes");
        accumulate_edges_pair<UNROLL, MODE>(p, beg0, end0, lane, acc[0], c0, 0.f, s0);
      } else {
#pragma unroll
        for (int k = 0; k < NACC; ++k) zero_vec(acc[k]);
        accumulate_edges<VEC, GROUP, NACC, UNROLL, MODE>(p, beg0, end0, 0, 1, gl, gmask, acc, c0, s0);
      }
      write_row<VEC, GROUP, NACC>(p, row0, gl, end0 > beg0, r0, acc, rmw, old);
    }
    slot0 = slot1; row0 = row1; beg0 = beg1; end0 = end1; c0 = c1; s0 = s1; r0 = r1;
    slot1 = slot2; row1 = row2; beg1 = beg2; end1 = end2; c1 = c2; m1 = m2;
    slot2 = slot3; row2 = row3; beg2 = beg3; end2 = end3;
  }
  finish();
}

template <int VEC, int GROUP, int NACC, int MODE, bool PAIR = false>
__global__ void __launch_bounds__(kBlockThreads) agg_rows_kernel(const AggParams p) {
  using T = typename VecT<VEC>::type;
  constexpr int GROUPS_PER_WARP = 32 / GROUP;
  const int lane = threadIdx.x & 31;
  const int gl = lane & (GROUP - 1);
  const unsigned gmask = (GROUP == 32) ? 0xffffffffu : (((1u << GROUP) - 1u) << (lane & ~(GROUP - 1)));
  const int warp = blockIdx.x * (kBlockThreads / 32) + (threadIdx.x >> 5);
  const int row = warp * GROUPS_PER_WARP + lane / GROUP;
  if (row >= p.num_rows) return;
  const int beg = __ldg(p.row_off + row);
  const int end = __ldg(p.row_off + row + 1);
  if (p.hub_threshold > 0 && (end - beg) > p.hub_threshold) return;  // hub kernel owns this row

  T acc[NACC];
  if constexpr (PAIR) {        // same summation order as the row-queue kernel: a row's bits do not depend on the graph size
    int c;
    float m, s;
    load_col<MODE>(p, beg, end, gl, c, m);
    load_scale<MODE>(p, beg, end, gl, c, m, s);
    accumulate_edges_pair<8, MODE>(p, beg, end, lane, acc[0], c, m, s);
  } else {
#pragma unroll
    for (int k = 0; k < NACC; ++k) zero_vec(acc[k]);
    accumulate_edges<VEC, GROUP, NACC, MODE>(p, beg, end, 0, 1, gl, gmask, acc);
  }

  const int orow = p.out_rows ? __ldg(p.out_rows + row) : row;
  const float r = p.rs ? __ldg(p.rs + orow) : 1.f;
  write_row<VEC, GROUP, NACC>(p, orow, gl, end > beg, r, acc);
  grid_dependency_wait();
}

// Hub rows (longer than hub_threshold) in two tiers.  The hub list is walked in chunks of kHubCluster
// entries by thread-block clusters of kHubCluster CTAs (16 warps each):
//   * a row of up to kClusterRowEdges edges is summed by ONE CTA (entry q of the chunk by CTA q), so a
//     cluster works on kHubCluster medium rows at once with no cluster-wide synchronisation;
//   * a longer row (10^4..10^5 edges on a power-law graph) is summed by the whole cluster: every
//     (CTA, warp, group) slot takes a strided share of the edge batches and the leader CTA adds the CTA
//     sums through distributed shared memory.
// Partials are reduced group->warp by shuffles, warp->CTA through shared memory, CTA->cluster over DSMEM,
// each level in a fixed order: deterministic, no atomics, no scratch buffer in HBM.  (One cluster per row
// for every hub row cost 10 us of latency chain + two cluster barriers per row: 0.66 ms for the 1077 hub
// rows of config 5; one CTA per row for every hub row leaves the chip idle behind a 10^5-edge row.)
constexpr int kHubCluster = 8;
constexpr int kClusterRowEdges = 8192;

template <int VEC, int GROUP, int NACC, int MODE>
__global__ void __cluster_dims__(kHubCluster, 1, 1) __launch_bounds__(kHubThreads)
    agg_hub_kernel(const AggParams p) {
  using T = typename VecT<VEC>::type;
  namespace cg = cooperative_groups;
  // The row kernel is launched behind this one as a programmatic dependent (see launch_agg): let it
  // start right away, the two kernels write disjoint rows.
  asm volatile("griddepcontrol.launch_dependents;");
  cg::cluster_group cluster = cg::this_cluster();
  constexpr int GROUPS_PER_WARP = 32 / GROUP;
  constexpr int WARPS = kHubThreads / 32;
  __shared__ T partial[WARPS][GROUP * NACC];
  __shared__ T cta_sum[GROUP * NACC];
  __shared__ int chunk_row[kHubCluster], chunk_beg[kHubCluster], chunk_end[kHubCluster];
  const int lane = threadIdx.x & 31;
  const int wid = threadIdx.x >> 5;
  const int gl = lane & (GROUP - 1);
  const int gidx = lane / GROUP;
  const unsigned gmask = (GROUP == 32) ? 0xffffffffu : (((1u << GROUP) - 1u) << (lane & ~(GROUP - 1)));
  const int crank = static_cast<int>(cluster.block_rank());
  const int cluster_id = blockIdx.x / kHubCluster;
  const int n_clusters = gridDim.x / kHubCluster;
  const int n_hub = min(__ldg(p.hub_count), p.hub_capacity);

  // Sum edges of [beg,end) over `slots` cooperating (warp, group) slots starting at `slot`, then reduce
  // the CTA's partials into cta_sum (valid after the trailing __syncthreads()).
  auto cta_partial_sum = [&](int beg, int end, int slot, int slots) {
    T acc[NACC];
#pragma unroll
    for (int k = 0; k < NACC; ++k) zero_vec(acc[k]);
    accumulate_edges<VEC, GROUP, NACC, MODE>(p, beg, end, slot, slots, gl, gmask, acc);
#pragma unroll
    for (int o = GROUP; o < 32; o <<= 1) {        // groups of one warp -> lanes [0, GROUP)
#pragma unroll
      for (int k = 0; k < NACC; ++k) add_vec(acc[k], shfl_xor_vec<T>(acc[k], o));
    }
    if (lane < GROUP) {
#pragma unroll
      for (int k = 0; k < NACC; ++k) partial[wid][k * GROUP + lane] = acc[k];
    }
    __syncthreads();
    if (wid == 0 && lane < GROUP) {               // warps of this CTA, fixed order
#pragma unroll
      for (int k = 0; k < NACC; ++k) {
        T sum = partial[0][k * GROUP + lane];
        for (int w = 1; w < WARPS; ++w) add_vec(sum, partial[w][k * GROUP + lane]);
        cta_sum[k * GROUP + lane] = sum;
      }
    }
    __syncthreads();
  };
  auto write_hub_row = [&](int row, T (&sum)[NACC]) {   // warp 0, lanes [0, GROUP)
    const int orow = p.out_rows ? __ldg(p.out_rows + row) : row;
    const float r = p.rs ? __ldg(p.rs + orow) : 1.f;
    write_row<VEC, GROUP, NACC>(p, orow, lane, true, r, sum);
  };

  for (int chunk = cluster_id; chunk * kHubCluster < n_hub; chunk += n_clusters) {
    if (threadIdx.x < kHubCluster) {
      const int i = chunk * kHubCluster + threadIdx.x;
      int row = -1, beg = 0, end = 0;
      if (i < n_hub) {
        row = __ldg(p.hub_rows + i);
        beg = __ldg(p.row_off + row);
        end = __ldg(p.row_off + row + 1);
      }
      chunk_row[threadIdx.x] = row;
      chunk_beg[threadIdx.x] = beg;
      chunk_end[threadIdx.x] = end;
    }
    __syncthreads();
    // tier 1: this CTA's own entry of the chunk
    {
      const int row = chunk_row[crank], beg = chunk_beg[crank], end = chunk_end[crank];
      if (row >= 0 && (end - beg) <= kClusterRowEdges) {
        cta_partial_sum(beg, end, wid * GROUPS_PER_WARP + gidx, WARPS * GROUPS_PER_WARP);
        if (wid == 0 && lane < GROUP) {
          T sum[NACC];
#pragma unroll
          for (int k = 0; k < NACC; ++k) sum[k] = cta_sum[k * GROUP + lane];
          write_hub_row(row, sum);
        }
      }
    }
    // tier 2: entries too long for one CTA, by the whole cluster (same decision in every CTA)
    for (int q = 0; q < kHubCluster; ++q) {
      const int row = chunk_row[q], beg = chunk_beg[q], end = chunk_end[q];
      if (row < 0 || (end - beg) <= kClusterRowEdges) continue;
      cta_partial_sum(beg, end, (crank * WARPS + wid) * GROUPS_PER_WARP + gidx, kHubCluster * WARPS * GROUPS_PER_WARP);
      cluster.sync();                               // every CTA's cta_sum is written
      if (crank == 0 && wid == 0 && lane < GROUP) { // CTAs of the cluster, fixed order, over DSMEM
        T sum[NACC];
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
          sum[k] = cta_sum[k * GROUP + lane];
          for (int c = 1; c < kHubCluster; ++c) {
            const T* remote = cluster.map_shared_rank(cta_sum, c);
            add_vec(sum[k], remote[k * GROUP + lane]);
          }
        }
        write_hub_row(row, sum);
      }
      cluster.sync();                               // peers keep cta_sum alive until the leader has read it
    }
    __syncthreads();                                // chunk_* are rewritten by the next iteration
  }
}

// A/B switch while the pair form is being measured (STG_AGG_PAIR=0/1; read once).
inline bool pair_mode() {
  static const bool on = [] {
    const char* e = getenv("STG_AGG_PAIR");
    return e == nullptr || e[0] != '0';
  }();
  return on;
}

// Slots a warp draws from the global row queue at a time (STG_AGG_CHUNK; 0 = static block ranges; read once).
inline int queue_chunk() {
  static const int v = [] {
    const char* e = getenv("STG_AGG_CHUNK");
    const int c = e ? atoi(e) : 4;
    return c < 0 ? 0 : (c > 4096 ? 4096 : c);
  }();
  return v;
}

// Hub CTAs per SM (STG_HUB_GRID overrides; read once).  Two 512-thread hub CTAs fill an SM's register file, so the row
// kernel launched behind them as a programmatic dependent cannot become resident before they retire: on a large graph
// one hub CTA per SM leaves half of every SM to the row kernel from the start (config 5 forward / backward 2.139 /
// 2.211 ms against 2.161 / 2.302 ms); small launches keep two (the hub rows are their critical path).
inline int hub_grid_mult(int num_edges) {
  static const int v = [] {
    const char* e = getenv("STG_HUB_GRID");
    const int c = e ? atoi(e) : 0;
    return c < 0 ? 0 : (c > 4 ? 4 : c);
  }();
  return v > 0 ? v : (num_edges >= (1 << 24) ? 1 : 2);
}

template <int VEC, int GROUP, int NACC, int MODE>
int launch_agg(const AggParams& p, cudaStream_t stream) {
  constexpr int rows_per_block = (kBlockThreads / 32) * (32 / GROUP);
  const int blocks = (p.num_rows + rows_per_block - 1) / rows_per_block;
  // Hub rows first: one cluster per row, at most one CTA per SM; the row kernel then fills the rest of
  // every SM instead of waiting for the last hub row (0.27 ms of a 3.5 ms launch on config 5).
  const bool hubs = p.hub_threshold > 0 && p.hub_rows != nullptr;
  // Small graphs gain nothing from the overlap and a programmatic edge costs extra inside a captured CUDA
  // graph (config 2, 1446 aggregations per epoch: 190 ms against 158 ms), so they keep plain stream order.
  const bool overlap = hubs && p.num_edges >= (1 << 18);
  if (hubs) {
    agg_hub_kernel<VEC, GROUP, NACC, MODE><<<hub_grid_mult(p.num_edges) * (sm_count() / kHubCluster) * kHubCluster, kHubThreads, 0, stream>>>(p);
    STG_LAUNCH_CHECK("agg_hub_kernel");
  }
  if (blocks > 0) {
    // A small graph (fewer rows than two waves of warps) keeps one row per warp: the queue kernel would put 256 rows
    // on each of a handful of SMs (Cora shape, F=100: 35 us against 7 us).
    const bool queue = p.num_rows >= 2 * sm_count() * 4 * (kBlockThreads / 32);
    bool launched = false;
    if constexpr (GROUP == 32 && MODE != kParts) if (queue) {
      launched = true;
      // measured on config 5 (F=100 / 128): 3.48 / 3.34 ms against 3.99 / 3.88 ms for one row per warp;
      // 4 resident blocks per SM beat 3 (4.2 ms) and 2 (5.2 ms), 5..8 with a shorter unroll do not help.
      constexpr int MINB = 4;           // 8 / NACC neighbour rows in flight per lane keep this at <= 64 registers
      // 32 rows per warp also on a 1/8 row slice of config 5 (306 K rows, two waves of blocks): 16 / 8 / 4 rows per
      // warp measured 0.32 / 0.35 / 0.39 ms against 0.316 ms -- the queue's balancing beats finer block granularity.
      constexpr int kRowsPerWarp = 32;
      constexpr int slots_per_block = (kBlockThreads / 32) * kRowsPerWarp;
      const int pblocks = (p.num_rows + slots_per_block - 1) / slots_per_block;
      // global row queue (the view carries its counters): resident blocks only, warps draw chunks of queue_chunk() slots
      const bool gq = p.queue != nullptr && queue_chunk() > 0;
      const int gblocks = std::min(sm_count() * MINB, (p.num_rows + 7) / 8);
      if constexpr (VEC == 4 && NACC == 1) {
        if (p.width > 64 && pair_mode()) {
          if (gq) {
            STG_CUDA(launch_overlapped(agg_rows_pipe_kernel<VEC, GROUP, NACC, MINB, 8, MODE, true, true>, gblocks, kBlockThreads,
                                       stream, overlap, p, queue_chunk()));
          } else {
            STG_CUDA(launch_overlapped(agg_rows_pipe_kernel<VEC, GROUP, NACC, MINB, 8, MODE, true>, pblocks, kBlockThreads,
                                       stream, overlap, p, slots_per_block));
          }
          STG_LAUNCH_CHECK("agg_rows_pipe_kernel (pair)");
          return STG_OK;
        }
      }
      if (gq) {
        STG_CUDA(launch_overlapped(agg_rows_pipe_kernel<VEC, GROUP, NACC, MINB, 8 / NACC, MODE, false, true>, gblocks,
                                   kBlockThreads, stream, overlap, p, queue_chunk()));
      } else {
        STG_CUDA(launch_overlapped(agg_rows_pipe_kernel<VEC, GROUP, NACC, MINB, 8 / NACC, MODE>, pblocks, kBlockThreads, stream,
                                   overlap, p, slots_per_block));
      }
    }
    if constexpr (GROUP == 32 && VEC == 4 && NACC == 1 && MODE != kParts) {
      if (!launched && p.width > 64 && pair_mode()) {
        STG_CUDA(launch_overlapped(agg_rows_kernel<VEC, GROUP, NACC, MODE, true>, blocks, kBlockThreads, stream, overlap, p));
        launched = true;
      }
    }
    if (!launched) {
      // narrow rows (several rows per warp): the lane groups of a warp diverge and the queue costs
      // more than it saves (F=64: 3.0 ms against 2.66 ms)
      STG_CUDA(launch_overlapped(agg_rows_kernel<VEC, GROUP, NACC, MODE>, blocks, kBlockThreads, stream, overlap, p));
    }
    STG_LAUNCH_CHECK("agg_rows_kernel");
  }
  return STG_OK;
}

inline bool narrow_vec2() {
  static const bool v = [] {
    const char* e = getenv("STG_AGG_NARROW_VEC2");
    return e ? atoi(e) != 0 : true;
  }();
  return v;
}

template <int VEC, int MODE>
int dispatch_group(const AggParams& p, cudaStream_t stream, int avg_degree) {
  const int nvec = p.width / VEC;
  // (A 8-lane x 4-chunk geometry for short rows was measured for the halo-source pass: slower, 0.40 vs 0.28 ms.)
  (void)avg_degree;
  if (nvec <= 1) return launch_agg<VEC, 1, 1, MODE>(p, stream);
  if (nvec <= 2) return launch_agg<VEC, 2, 1, MODE>(p, stream);
  if (nvec <= 4) return launch_agg<VEC, 4, 1, MODE>(p, stream);
  if (nvec <= 8) return launch_agg<VEC, 8, 1, MODE>(p, stream);
  if (nvec <= 16) return launch_agg<VEC, 16, 1, MODE>(p, stream);
  if (nvec <= 32) return launch_agg<VEC, 32, 1, MODE>(p, stream);
  if (nvec <= 64) return launch_agg<VEC, 32, 2, MODE>(p, stream);
  return launch_agg<VEC, 32, 4, MODE>(p, stream);
}

// {column, nbr_scale[column] * edge_scale[eid]} of every CSR slot, in CSR order (same product order as
// load_scale<kPlain>, so the packed and the plain path give bit-identical sums).
__global__ void __launch_bounds__(256) pack_edge_meta_kernel(const AggParams p, int2* __restrict__ meta) {
  const int stride = gridDim.x * blockDim.x;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < p.num_edges; e += stride) {
    const int c = ld_stream(p.col + e);
    float sc = 1.f;
    if (p.ns) sc = __ldg(p.ns + c);
    if (p.es) {
      const int eid = p.eids_identity ? e : (ld_stream(p.eids + e) - p.eid_base);
      sc *= __ldg(p.es + eid);
    }
    __stcs(meta + e, make_int2(c, __float_as_int(sc)));
  }
}

}  // namespace

int agg_scaled_sum_device(const StgCsrView* g, const float* x, int32_t feat, const float* ns,
                          const float* es, const float* rs, float* out, cudaStream_t stream,
                          int nparts = 0, const float* const* parts = nullptr, const int32_t* bounds = nullptr,
                          int accumulate = 0, const int32_t* out_rows = nullptr, const StgEdgeMeta* meta = nullptr,
                          int x_ld = 0, int out_ld = 0) {
  AggParams p;
  p.out_rows = out_rows;
  p.meta = reinterpret_cast<const int2*>(meta);
  p.queue = g->work_queue;
  p.accumulate = accumulate;
  p.nparts = nparts;
  for (int q = 0; q < STG_MAX_PARTS; ++q) p.xs[q] = q < nparts ? parts[q] : nullptr;
  for (int q = 0; q <= STG_MAX_PARTS; ++q) p.bounds[q] = (nparts > 0 && q <= nparts) ? bounds[q] : 0;
  p.row_off = g->row_offset;
  p.col = g->column_indices;
  p.eids = g->eids;
  p.hub_rows = g->hub_rows;
  p.hub_count = g->hub_count;
  p.num_rows = g->num_nodes;
  p.num_edges = g->num_edges;
  p.eid_base = g->eid_base;
  p.eids_identity = g->eids_identity;
  p.hub_threshold = (g->hub_rows && g->hub_count) ? g->hub_threshold : 0;
  p.hub_capacity = g->hub_capacity;
  p.ld = x_ld > 0 ? x_ld : feat;
  p.ld_out = out_ld > 0 ? out_ld : feat;
  p.ns = ns;
  p.es = es;
  p.rs = rs;
  bool al16 = aligned16(out), al8 = aligned8(out);
  if (nparts == 0) {
    al16 = al16 && aligned16(x);
    al8 = al8 && aligned8(x);
  }
  for (int q = 0; q < nparts; ++q) {
    al16 = al16 && aligned16(parts[q]);
    al8 = al8 && aligned8(parts[q]);
  }
  int vec = 1;
  if (feat % 4 == 0 && p.ld % 4 == 0 && p.ld_out % 4 == 0 && al16) vec = 4;
  else if (feat % 2 == 0 && p.ld % 2 == 0 && p.ld_out % 2 == 0 && al8) vec = 2;
  // 33..64 floats per row with 128-bit loads are two rows per warp on the static schedule; 64-bit loads make them one
  // row per warp, which runs on the global row queue (STG_AGG_NARROW_VEC2=0 keeps the 128-bit form)
  if (vec == 4 && feat > 32 && feat <= 64 && nparts == 0 && narrow_vec2() && g->work_queue != nullptr &&
      g->num_nodes >= 2 * sm_count() * 4 * (kBlockThreads / 32))
    vec = 2;
  const int chunk = 32 * 4 * vec;  // widest tile one launch covers
  for (int f0 = 0; f0 < feat; f0 += chunk) {
    p.x = x ? x + f0 : nullptr;
    for (int q = 0; q < nparts; ++q) p.xs[q] = parts[q] + f0;
    p.out = out + f0;
    p.width = min(chunk, feat - f0);
    int rc;
    const int avg_degree = g->num_nodes > 0 ? g->num_edges / g->num_nodes : -1;
    if (nparts > 0) {
      if (vec == 4) rc = dispatch_group<4, kParts>(p, stream, avg_degree);
      else if (vec == 2) rc = dispatch_group<2, kParts>(p, stream, avg_degree);
      else rc = dispatch_group<1, kParts>(p, stream, avg_degree);
    } else if (meta != nullptr) {
      if (vec == 4) rc = dispatch_group<4, kPacked>(p, stream, avg_degree);
      else if (vec == 2) rc = dispatch_group<2, kPacked>(p, stream, avg_degree);
      else rc = dispatch_group<1, kPacked>(p, stream, avg_degree);
    } else {
      if (vec == 4) rc = dispatch_group<4, kPlain>(p, stream, avg_degree);
      else if (vec == 2) rc = dispatch_group<2, kPlain>(p, stream, avg_degree);
      else rc = dispatch_group<1, kPlain>(p, stream, avg_degree);
    }
    if (rc != STG_OK) return rc;
  }
  return STG_OK;
}

}  // namespace stg

using namespace stg;

STG_API int stg_agg_scaled_sum_f32(const StgCsrView* g, const float* x, int32_t feat,
                                      const float* nbr_scale, const float* edge_scale,
                                      const float* row_scale, float* out, void* stream) {
  int rc = validate_view(g, edge_scale != nullptr);
  if (rc != STG_OK) return rc;
  STG_CHECK_ARG(feat > 0, "feat must be positive (got %d)", feat);
  if (g->num_nodes == 0) return STG_OK;
  STG_CHECK_ARG(x != nullptr && out != nullptr, "x / out is NULL");
  STG_CHECK_ARG(x != out, "x and out must not alias");
  return agg_scaled_sum_device(g, x, feat, nbr_scale, edge_scale, row_scale, out, as_stream(stream));
}

static int agg_host_enqueue(const StgCsrView* g, const float* x_host, int32_t feat, const float* nbr_scale_host,
                            const float* edge_scale_host, const float* row_scale_host, float* out_host,
                            void* dev_scratch, size_t dev_scratch_bytes, void* stream, bool synchronize) {
  int rc = validate_view(g, edge_scale_host != nullptr);
  if (rc != STG_OK) return rc;
  STG_CHECK_ARG(feat > 0, "feat must be positive (got %d)", feat);
  if (g->num_nodes == 0) return STG_OK;
  STG_CHECK_ARG(x_host && out_host && dev_scratch, "host buffers / scratch must not be NULL");
  const size_t n = static_cast<size_t>(g->num_nodes), e = static_cast<size_t>(g->num_edges);
  const size_t nf = align_up(n * feat, 4), n4 = align_up(n, 4), e4 = align_up(e, 4);
  const size_t need = (2 * nf + 2 * n4 + e4) * sizeof(float);
  if (dev_scratch_bytes < need) {
    set_error("device scratch too small: %zu bytes given, %zu needed", dev_scratch_bytes, need);
    return STG_ERR_WORKSPACE_TOO_SMALL;
  }
  cudaStream_t s = as_stream(stream);
  float* dx = static_cast<float*>(dev_scratch);
  float* dout = dx + nf;
  float* dns = dout + nf;
  float* drs = dns + n4;
  float* des = drs + n4;
  STG_CUDA(cudaMemcpyAsync(dx, x_host, n * feat * sizeof(float), cudaMemcpyHostToDevice, s));
  if (nbr_scale_host) STG_CUDA(cudaMemcpyAsync(dns, nbr_scale_host, n * sizeof(float), cudaMemcpyHostToDevice, s));
  if (row_scale_host) STG_CUDA(cudaMemcpyAsync(drs, row_scale_host, n * sizeof(float), cudaMemcpyHostToDevice, s));
  if (edge_scale_host) STG_CUDA(cudaMemcpyAsync(des, edge_scale_host, e * sizeof(float), cudaMemcpyHostToDevice, s));
  rc = agg_scaled_sum_device(g, dx, feat, nbr_scale_host ? dns : nullptr, edge_scale_host ? des : nullptr,
                             row_scale_host ? drs : nullptr, dout, s);
  if (rc != STG_OK) return rc;
  STG_CUDA(cudaMemcpyAsync(out_host, dout, n * feat * sizeof(float), cudaMemcpyDeviceToHost, s));
  if (synchronize) STG_CUDA(cudaStreamSynchronize(s));
  return STG_OK;
}

STG_API int stg_agg_scaled_sum_f32_host(const StgCsrView* g, const float* x_host, int32_t feat,
                                        const float* nbr_scale_host, const float* edge_scale_host,
                                        const float* row_scale_host, float* out_host,
                                        void* dev_scratch, size_t dev_scratch_bytes, void* stream) {
  return agg_host_enqueue(g, x_host, feat, nbr_scale_host, edge_scale_host, row_scale_host, out_host, dev_scratch,
                          dev_scratch_bytes, stream, true);
}

STG_API int stg_agg_scaled_sum_f32_host_async(const StgCsrView* g, const float* x_host, int32_t feat,
                                              const float* nbr_scale_host, const float* edge_scale_host,
                                              const float* row_scale_host, float* out_host,
                                              void* dev_scratch, size_t dev_scratch_bytes, void* stream) {
  return agg_host_enqueue(g, x_host, feat, nbr_scale_host, edge_scale_host, row_scale_host, out_host, dev_scratch,
                          dev_scratch_bytes, stream, false);
}

STG_API int stg_agg_scaled_sum_parts_f32(const StgCsrView* g, const float* const* x_parts, const int32_t* part_bounds,
                                         int32_t num_parts, int32_t feat, const float* nbr_scale,
                                         const float* edge_scale, const float* row_scale, float* out, void* stream) {
  int rc = validate_view(g, edge_scale != nullptr);
  if (rc != STG_OK) return rc;
  STG_CHECK_ARG(feat > 0, "feat must be positive (got %d)", feat);
  STG_CHECK_ARG(num_parts >= 1 && num_parts <= STG_MAX_PARTS, "num_parts must be in [1, %d] (got %d)", STG_MAX_PARTS,
                num_parts);
  STG_CHECK_ARG(x_parts && part_bounds && out, "NULL argument");
  for (int q = 0; q < num_parts; ++q) {
    STG_CHECK_ARG(part_bounds[q] <= part_bounds[q + 1], "part_bounds must be non-decreasing");
    STG_CHECK_ARG(x_parts[q] != nullptr || part_bounds[q] == part_bounds[q + 1], "x_parts[%d] is NULL", q);
  }
  STG_CHECK_ARG(part_bounds[0] == 0, "part_bounds[0] must be 0");
  if (g->num_nodes == 0) return STG_OK;
  return agg_scaled_sum_device(g, nullptr, feat, nbr_scale, edge_scale, row_scale, out, as_stream(stream), num_parts,
                               x_parts, part_bounds);
}

STG_API int stg_agg_scaled_sum_accum_f32(const StgCsrView* g, const float* x, int32_t feat, const float* nbr_scale,
                                         const float* edge_scale, const float* row_scale, float* out, void* stream) {
  int rc = validate_view(g, edge_scale != nullptr);
  if (rc != STG_OK) return rc;
  STG_CHECK_ARG(feat > 0, "feat must be positive (got %d)", feat);
  if (g->num_nodes == 0) return STG_OK;
  STG_CHECK_ARG(x != nullptr && out != nullptr, "x / out is NULL");
  STG_CHECK_ARG(x != out, "x and out must not alias");
  return agg_scaled_sum_device(g, x, feat, nbr_scale, edge_scale, row_scale, out, as_stream(stream), 0, nullptr, nullptr, 1);
}

STG_API int stg_agg_scaled_sum_rows_f32(const StgCsrView* g, const int32_t* out_rows, const float* x, int32_t feat,
                                        const float* nbr_scale, const float* edge_scale, const float* row_scale,
                                        float* out, int32_t accumulate, void* stream) {
  int rc = validate_view(g, edge_scale != nullptr);
  if (rc != STG_OK) return rc;
  STG_CHECK_ARG(feat > 0, "feat must be positive (got %d)", feat);
  STG_CHECK_ARG(accumulate >= 0 && accumulate <= 2, "accumulate must be 0, 1 or 2 (got %d)", accumulate);
  if (g->num_nodes == 0) return STG_OK;
  STG_CHECK_ARG(out_rows != nullptr, "out_rows is NULL");
  STG_CHECK_ARG(x != nullptr && out != nullptr, "x / out is NULL");
  STG_CHECK_ARG(x != out, "x and out must not alias");
  return agg_scaled_sum_device(g, x, feat, nbr_scale, edge_scale, row_scale, out, as_stream(stream), 0, nullptr, nullptr,
                               accumulate, out_rows);
}

STG_API int stg_agg_scaled_sum_red_f32(const StgCsrView* g, const float* x, int32_t feat, const float* nbr_scale,
                                       const float* edge_scale, const float* row_scale, float* out, void* stream) {
  int rc = validate_view(g, edge_scale != nullptr);
  if (rc != STG_OK) return rc;
  STG_CHECK_ARG(feat > 0, "feat must be positive (got %d)", feat);
  if (g->num_nodes == 0) return STG_OK;
  STG_CHECK_ARG(x != nullptr && out != nullptr, "x / out is NULL");
  STG_CHECK_ARG(x != out, "x and out must not alias");
  return agg_scaled_sum_device(g, x, feat, nbr_scale, edge_scale, row_scale, out, as_stream(stream), 0, nullptr, nullptr, 2);
}

STG_API int stg_csr_pack_edge_meta_f32(const StgCsrView* g, const float* nbr_scale, const float* edge_scale,
                                       StgEdgeMeta* meta, void* stream) {
  int rc = validate_view(g, edge_scale != nullptr);
  if (rc != STG_OK) return rc;
  if (g->num_edges == 0) return STG_OK;
  STG_CHECK_ARG(meta != nullptr && aligned8(meta), "meta must be a non-NULL, 8-byte aligned device pointer");
  AggParams p = {};
  p.col = g->column_indices;
  p.eids = g->eids;
  p.num_edges = g->num_edges;
  p.eid_base = g->eid_base;
  p.eids_identity = g->eids_identity;
  p.ns = nbr_scale;
  p.es = edge_scale;
  const int blocks = static_cast<int>(std::min<int64_t>((static_cast<int64_t>(g->num_edges) + 255) / 256, 8 * sm_count()));
  pack_edge_meta_kernel<<<blocks, 256, 0, as_stream(stream)>>>(p, reinterpret_cast<int2*>(meta));
  STG_LAUNCH_CHECK("pack_edge_meta_kernel");
  return STG_OK;
}

STG_API int stg_agg_packed_sum_strided_f32(const StgCsrView* g, const StgEdgeMeta* meta, const float* x, int32_t feat,
                                           int32_t x_ld, const float* row_scale, float* out, int32_t out_ld,
                                           int32_t accumulate, void* stream) {
  int rc = validate_view(g, false);
  if (rc != STG_OK) return rc;
  STG_CHECK_ARG(feat > 0, "feat must be positive (got %d)", feat);
  STG_CHECK_ARG(x_ld >= feat && out_ld >= feat, "row strides (%d, %d) must be >= feat (%d)", x_ld, out_ld, feat);
  STG_CHECK_ARG(accumulate >= 0 && accumulate <= 2, "accumulate must be 0, 1 or 2 (got %d)", accumulate);
  if (g->num_nodes == 0) return STG_OK;
  STG_CHECK_ARG(g->num_edges == 0 || (meta != nullptr && aligned8(meta)),
                "meta must be a non-NULL, 8-byte aligned device pointer");
  STG_CHECK_ARG(x != nullptr && out != nullptr, "x / out is NULL");
  STG_CHECK_ARG(x != out, "x and out must not alias");
  // an empty graph has nothing to read through meta: the plain path writes the zero rows
  return agg_scaled_sum_device(g, x, feat, nullptr, nullptr, row_scale, out, as_stream(stream), 0, nullptr, nullptr,
                               accumulate, nullptr, g->num_edges == 0 ? nullptr : meta, x_ld, out_ld);
}

STG_API int stg_agg_packed_sum_f32(const StgCsrView* g, const StgEdgeMeta* meta, const float* x, int32_t feat,
                                   const float* row_scale, float* out, int32_t accumulate, void* stream) {
  return stg_agg_packed_sum_strided_f32(g, meta, x, feat, feat, row_scale, out, feat, accumulate, stream);
}

STG_API int stg_agg_packed_sum_rows_f32(const StgCsrView* g, const StgEdgeMeta* meta, const int32_t* out_rows,
                                        const float* x, int32_t feat, const float* row_scale, float* out,
                                        int32_t accumulate, void* stream) {
  int rc = validate_view(g, false);
  if (rc != STG_OK) return rc;
  STG_CHECK_ARG(feat > 0, "feat must be positive (got %d)", feat);
  STG_CHECK_ARG(accumulate >= 0 && accumulate <= 2, "accumulate must be 0, 1 or 2 (got %d)", accumulate);
  if (g->num_nodes == 0) return STG_OK;
  STG_CHECK_ARG(g->num_edges == 0 || (meta != nullptr && aligned8(meta)),
                "meta must be a non-NULL, 8-byte aligned device pointer");
  STG_CHECK_ARG(x != nullptr && out != nullptr, "x / out is NULL");
  STG_CHECK_ARG(x != out, "x and out must not alias");
  return agg_scaled_sum_device(g, x, feat, nullptr, nullptr, row_scale, out, as_stream(stream), 0, nullptr, nullptr,
                               accumulate, out_rows, g->num_edges == 0 ? nullptr : meta);
}
