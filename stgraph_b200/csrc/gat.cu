// Fused edge-softmax attention aggregation (GAT) for sm_100a.
//
// Reference: GATConv's vertex program (stgraph/nn/pytorch/static/gat_conv.py:48-56) compiles to two
// forward kernels with a materialised [E,H,1] score tensor (K0: scores + row sums, K1: weighted sum)
// and one backward kernel that accumulates d_el / d_er with per-lane atomicAdd, E*H*D of them inside
// the edge loop (SURVEY.md appendix A.3).  As shipped the program even degenerates to a mean (trap
// T2); the stock program therefore runs through the generic VM kernel, bit-faithful to the trace.
// These kernels are the genuine edge softmax a fixed program would compute:
//   forward : ONE pass per destination row with an online softmax (running max / sum per head),
//             nothing of size E is written; row max and row sum ([N,H]) are kept for backward.
//   backward: alpha is recomputed from (el, er, max, sum).  Pass A walks the in-edge CSR
//             (destination-parallel): dot[v,h] = <dout[v,h,:], out[v,h,:]>, d_er.  Pass B walks the
//             out-edge CSR (source-parallel): d_feat, d_el.  Every output row is owned by one lane
//             group (or one block for hub rows): no atomics, deterministic.
// A lane group owns a row; a lane owns VEC consecutive floats of the flattened [H*D] row per chunk,
// so one neighbour row is one coalesced (128-bit when D % 4 == 0) load; UNROLL neighbour rows are
// loaded before any of them is consumed (the online-softmax update is applied per batch, so the
// running max does not serialise the loads).  Rows longer than the view's hub threshold go to a
// block-per-row kernel: 8 warps take strided batches and their (max, sum, acc) partials are merged
// in a fixed order through shuffles + shared memory.
// HBM-roofline kernels; algorithmic bytes: fwd 4*(2*N*H*D + 4*N*H + E + N+1),
// bwd 4*(4*N*H*D + 6*N*H + 2*(E+N+1)).
#include "common.cuh"
#include "h16.cuh"

#include <cooperative_groups.h>

#include <algorithm>
#include <cstdlib>
#include <type_traits>

namespace stg {
namespace {

constexpr int kGatThreads = 256;
constexpr int kGatHubThreads = 256;   // 8 warps per hub CTA: a 130-edge row has 5 batches, 16 warps would mostly wait at the barrier

template <int VEC>
__device__ __forceinline__ typename VecT<VEC>::type ldv(const float* p) {
  using T = typename VecT<VEC>::type;
  return __ldg(reinterpret_cast<const T*>(p));
}
template <int VEC>
__device__ __forceinline__ void stv(float* p, typename VecT<VEC>::type v) {
  using T = typename VecT<VEC>::type;
  *reinterpret_cast<T*>(p) = v;
}
// feat / d_feat elements of storage type FT (float, __nv_bfloat16, __half): VEC of them per lane, one 8- or 2-byte
// access for 16-bit rows, widened to fp32 and rounded to nearest even on the store.  The forward edge loop keeps a
// gathered row in its loaded form (FtRaw) until the batch's arithmetic: widening right after the load, inside the
// `if (L.act[k])` of the batch, made the compiler branch around each load and wait for it before issuing the next one
// (config 3: 0.194 ms against 0.152 ms for fp32 rows).  Backward pass A widens on load: it was not slower that way, and
// with the later widening its d_er no longer matched the fp32 kernel's bit for bit.
template <int VEC, typename FT> struct FtRaw { using type = typename Raw<VEC>::type; };
template <int VEC> struct FtRaw<VEC, float> { using type = typename VecT<VEC>::type; };
using stg::zero_vec;
__device__ __forceinline__ void zero_vec(uint2& a) { a = make_uint2(0u, 0u); }
__device__ __forceinline__ void zero_vec(unsigned short& a) { a = 0; }

template <int VEC, typename FT>
__device__ __forceinline__ typename FtRaw<VEC, FT>::type ldraw(const FT* p) {
  if constexpr (std::is_same_v<FT, float>) return ldv<VEC>(p);
  else return __ldg(reinterpret_cast<const typename Raw<VEC>::type*>(p));
}
template <int VEC, typename FT>
__device__ __forceinline__ typename VecT<VEC>::type widen(const typename FtRaw<VEC, FT>::type& r) {
  if constexpr (std::is_same_v<FT, float>) {
    return r;
  } else {
    float f[VEC];
    unpack<FT, VEC>(r, f);
    if constexpr (VEC == 4) return make_float4(f[0], f[1], f[2], f[3]);
    else return f[0];
  }
}
template <int VEC, typename FT>
__device__ __forceinline__ typename VecT<VEC>::type ldf(const FT* p) {
  return widen<VEC, FT>(ldraw<VEC>(p));
}
template <int VEC, typename FT>
__device__ __forceinline__ void stf(FT* p, typename VecT<VEC>::type v) {
  if constexpr (std::is_same_v<FT, float>) {
    stv<VEC>(p, v);
  } else {
    float f[VEC];
    if constexpr (VEC == 4) f[0] = v.x, f[1] = v.y, f[2] = v.z, f[3] = v.w;
    else f[0] = v;
    *reinterpret_cast<typename Raw<VEC>::type*>(p) = pack<FT, VEC>(f);
  }
}
__device__ __forceinline__ float dotv(float a, float b) { return a * b; }
__device__ __forceinline__ float dotv(float2 a, float2 b) { return a.x * b.x + a.y * b.y; }
__device__ __forceinline__ float dotv(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
__device__ __forceinline__ float lrelu(float x, float slope) { return x > 0.f ? x : slope * x; }

__device__ __forceinline__ float shfl_xor_t(unsigned m, float v, int o) { return __shfl_xor_sync(m, v, o); }
__device__ __forceinline__ float2 shfl_xor_t(unsigned m, float2 v, int o) {
  return make_float2(__shfl_xor_sync(m, v.x, o), __shfl_xor_sync(m, v.y, o));
}
__device__ __forceinline__ float4 shfl_xor_t(unsigned m, float4 v, int o) {
  return make_float4(__shfl_xor_sync(m, v.x, o), __shfl_xor_sync(m, v.y, o), __shfl_xor_sync(m, v.z, o),
                     __shfl_xor_sync(m, v.w, o));
}

// FT: storage type of feat and d_feat; every other tensor, and all arithmetic, is fp32.
template <typename FT>
struct GatParams {
  using feat_t = FT;
  const int32_t* __restrict__ row_off;
  const int32_t* __restrict__ col;
  const int32_t* __restrict__ hub_rows;
  const int32_t* __restrict__ hub_count;
  int hub_threshold, hub_capacity;
  int* queue;            // global row queue of the view (StgCsrView::work_queue) or NULL
  int num_rows;
  int heads, dim, hd;        // hd = heads*dim
  int lph;                   // lanes per head inside a chunk (dim / VEC), power of two
  float slope;
  const float* __restrict__ el;     // [N,H]
  const float* __restrict__ er;     // [N,H]
  const FT* __restrict__ feat;      // [N,H,D]
  const float* __restrict__ out;    // [N,H,D]  (backward)
  const float* __restrict__ gout;   // [N,H,D]  (backward)
  float* __restrict__ row_max;      // [N,H]
  float* __restrict__ row_sum;      // [N,H]
  float* __restrict__ dot;          // [N,H]    (backward scratch)
  float* __restrict__ o_vec;        // forward: out; backward pass B: d_feat (FT elements, see gat_bwd_store)
  float* __restrict__ o_head;       // backward: d_er (pass A) / d_el (pass B)
};

template <int VEC, int GROUP, int NACC>
struct Lanes {
  int gl;
  unsigned gmask;
  int off[NACC], hk[NACC];
  bool act[NACC];
  template <class P>
  __device__ __forceinline__ void init(const P& p) {
    const int lane = threadIdx.x & 31;
    gl = lane & (GROUP - 1);
    gmask = (GROUP == 32) ? 0xffffffffu : (((1u << GROUP) - 1u) << (lane & ~(GROUP - 1)));
#pragma unroll
    for (int k = 0; k < NACC; ++k) {
      off[k] = (gl + k * GROUP) * VEC;
      act[k] = off[k] < p.hd;
      hk[k] = act[k] ? off[k] / p.dim : 0;
    }
  }
};

// sum over the lanes of one head (lph consecutive lanes, power of two)
__device__ __forceinline__ float head_sum(float v, int lph, unsigned gmask, int width) {
  for (int o = 1; o < lph; o <<= 1) v += __shfl_xor_sync(gmask, v, o, width);
  return v;
}

// neighbour rows in flight per lane: a row of n edges costs n / U dependent L2 round trips, and on a power-law
// graph the longest rows set the kernel time (config 3: 0.40 -> see profiles/r01_results.md)
template <int NACC> struct UnrollFor { static constexpr int value = NACC >= 4 ? 2 : (NACC == 2 ? 4 : 8); };
// the backward passes carry four per-edge scalars next to each neighbour row: 8 in flight would cost occupancy
template <int NACC> struct UnrollBwd { static constexpr int value = NACC >= 4 ? 2 : 4; };

// Calls body(integral_constant<G>, j) over [0, n) with G = U for every full group and ONE exactly-sized group for the
// tail: a row of 7 edges is one batch of 7 loads (one L2 round trip), not 4 + 2 + 1 (three dependent ones).
template <int U, class Body>
__device__ __forceinline__ void for_exact_groups(int n, Body&& body) {
  int j = 0;
  for (; j + U <= n; j += U) body(std::integral_constant<int, U>{}, j);
  if constexpr (U >= 2) {
    switch (n - j) {
      case 1: body(std::integral_constant<int, 1>{}, j); break;
      case 2: if constexpr (U > 2) body(std::integral_constant<int, 2>{}, j); break;
      case 3: if constexpr (U > 3) body(std::integral_constant<int, 3>{}, j); break;
      case 4: if constexpr (U > 4) body(std::integral_constant<int, 4>{}, j); break;
      case 5: if constexpr (U > 5) body(std::integral_constant<int, 5>{}, j); break;
      case 6: if constexpr (U > 6) body(std::integral_constant<int, 6>{}, j); break;
      case 7: if constexpr (U > 7) body(std::integral_constant<int, 7>{}, j); break;
      default: break;
    }
  }
}

// ---------------------------------------------------------------------------------- forward
template <int VEC, int GROUP, int NACC>
struct FwdState {
  using T = typename VecT<VEC>::type;
  float m[NACC], s[NACC];
  T acc[NACC];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int k = 0; k < NACC; ++k) {
      m[k] = -INFINITY;
      s[k] = 0.f;
      zero_vec(acc[k]);
    }
  }
  // merge another partial (online-softmax combine); safe when either side is still empty (m = -inf)
  __device__ __forceinline__ void merge(int k, float m2, float s2, T a2) {
    const float mm = fmaxf(m[k], m2);
    const float f1 = (m[k] == -INFINITY) ? 0.f : __expf(m[k] - mm);
    const float f2 = (m2 == -INFINITY) ? 0.f : __expf(m2 - mm);
    s[k] = s[k] * f1 + s2 * f2;
    scale_vec(acc[k], f1);
    fma_vec(acc[k], f2, a2);
    m[k] = mm;
  }
};

template <int VEC, int GROUP, int NACC, class P>
__device__ __forceinline__ void gat_fwd_edges(const P& p, const Lanes<VEC, GROUP, NACC>& L, int row, int beg,
                                              int end, int first_batch, int batch_step,
                                              FwdState<VEC, GROUP, NACC>& st, int nx_c) {
  using FT = typename P::feat_t;
  constexpr int U = UnrollFor<NACC>::value;
  float erk[NACC];
#pragma unroll
  for (int k = 0; k < NACC; ++k) erk[k] = L.act[k] ? __ldg(p.er + static_cast<size_t>(row) * p.heads + L.hk[k]) : 0.f;
  int base = beg + first_batch * GROUP;
  for (; base < end; base += batch_step * GROUP) {
    const int n = min(GROUP, end - base);
    const int my_c = nx_c;
    {                                             // column indices of the next batch, one batch ahead
      const int nb = base + batch_step * GROUP + L.gl;
      nx_c = (nb < end) ? ld_stream(p.col + nb) : 0;
    }
    // Exactly-sized groups (8, then 4 / 2 / 1 for the tail): no padding edges, so no per-edge predicates, and a
    // 3-edge row costs 3 edges of instructions, not 8 (most rows of a power-law graph are that short: the row
    // kernel was issue-bound at 545 warp instructions per row, profiles/r01_results.md).
    auto group = [&](auto uu, int j) {
      constexpr int UU = decltype(uu)::value;
      float sc[UU][NACC];
      typename FtRaw<VEC, FT>::type v[UU][NACC];
#pragma unroll
      for (int u = 0; u < UU; ++u) {
        const int c = __shfl_sync(L.gmask, my_c, j + u, GROUP);
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
          sc[u][k] = -INFINITY;
          zero_vec(v[u][k]);
          if (L.act[k]) {
            sc[u][k] = lrelu(__ldg(p.el + static_cast<size_t>(c) * p.heads + L.hk[k]) + erk[k], p.slope);
            v[u][k] = ldraw<VEC>(p.feat + static_cast<size_t>(c) * p.hd + L.off[k]);
          }
        }
      }
#pragma unroll
      for (int k = 0; k < NACC; ++k) {
        if (!L.act[k]) continue;
        float mb = sc[0][k];
#pragma unroll
        for (int u = 1; u < UU; ++u) mb = fmaxf(mb, sc[u][k]);
        if (mb > st.m[k]) {                       // new running max: rescale what has been accumulated
          const float r = __expf(st.m[k] - mb);   // exp(-inf) = 0 on the first group
          st.s[k] *= r;
          scale_vec(st.acc[k], r);
          st.m[k] = mb;
        }
#pragma unroll
        for (int u = 0; u < UU; ++u) {
          const float pe = __expf(sc[u][k] - st.m[k]);
          st.s[k] += pe;
          fma_vec(st.acc[k], pe, widen<VEC, FT>(v[u][k]));
        }
      }
    };
    for_exact_groups<U>(n, group);
  }
}

// columns of the first batch a lane group visits (the pipelined kernels load them one row ahead instead)
template <int GROUP, class P>
__device__ __forceinline__ int first_cols(const P& p, int beg, int end, int first_batch, int gl) {
  const int e = beg + first_batch * GROUP + gl;
  return (e < end) ? ld_stream(p.col + e) : 0;
}

template <int VEC, int GROUP, int NACC, class P>
__device__ __forceinline__ void gat_fwd_store(const P& p, const Lanes<VEC, GROUP, NACC>& L, int row,
                                              bool nonempty, FwdState<VEC, GROUP, NACC>& st) {
#pragma unroll
  for (int k = 0; k < NACC; ++k) {
    if (!L.act[k]) continue;
    const float inv = st.s[k] > 0.f ? 1.f / st.s[k] : 0.f;
    scale_vec(st.acc[k], inv);
    stv<VEC>(p.o_vec + static_cast<size_t>(row) * p.hd + L.off[k], st.acc[k]);
    if (L.off[k] % p.dim == 0) {
      p.row_max[static_cast<size_t>(row) * p.heads + L.hk[k]] = nonempty ? st.m[k] : 0.f;
      p.row_sum[static_cast<size_t>(row) * p.heads + L.hk[k]] = st.s[k];
    }
  }
}

template <typename FT, int VEC, int GROUP, int NACC>
__global__ void __launch_bounds__(kGatThreads) gat_fwd_kernel(const GatParams<FT> p) {
  Lanes<VEC, GROUP, NACC> L;
  L.init(p);
  const int warp = blockIdx.x * (kGatThreads / 32) + (threadIdx.x >> 5);
  const int row = warp * (32 / GROUP) + (threadIdx.x & 31) / GROUP;
  if (row < p.num_rows) {
    const int beg = __ldg(p.row_off + row), end = __ldg(p.row_off + row + 1);
    if (!(p.hub_threshold > 0 && (end - beg) > p.hub_threshold)) {   // else: the hub kernel owns this row
      FwdState<VEC, GROUP, NACC> st;
      st.init();
      gat_fwd_edges<VEC, GROUP, NACC>(p, L, row, beg, end, 0, 1, st, first_cols<GROUP>(p, beg, end, 0, L.gl));
      gat_fwd_store<VEC, GROUP, NACC>(p, L, row, end > beg, st);
    }
  }
  grid_dependency_wait();
}

// --------------------------------------------------------------------------------- backward
// SRC_PARALLEL = false: pass A (rows = destinations): dot, d_er.
// SRC_PARALLEL = true : pass B (rows = sources): d_feat, d_el.
template <int VEC, int GROUP, int NACC>
struct BwdState {
  using T = typename VecT<VEC>::type;
  T cen[NACC], accv[NACC];
  float acch[NACC], c_a[NACC], c_m[NACC], c_inv[NACC], c_dot[NACC];
};

template <int VEC, int GROUP, int NACC, bool SRC_PARALLEL, class P>
__device__ __forceinline__ void gat_bwd_prologue(const P& p, const Lanes<VEC, GROUP, NACC>& L, int row,
                                                 BwdState<VEC, GROUP, NACC>& st, bool write_dot) {
  const size_t rh = static_cast<size_t>(row) * p.heads;
#pragma unroll
  for (int k = 0; k < NACC; ++k) {
    st.acch[k] = 0.f;
    zero_vec(st.accv[k]);
    zero_vec(st.cen[k]);
    st.c_a[k] = st.c_m[k] = st.c_inv[k] = st.c_dot[k] = 0.f;
    float part = 0.f;
    const size_t ro = static_cast<size_t>(row) * p.hd + L.off[k];
    if (L.act[k]) {
      if (SRC_PARALLEL) {
        st.cen[k] = ldf<VEC>(p.feat + ro);
        st.c_a[k] = __ldg(p.el + rh + L.hk[k]);
      } else {
        st.cen[k] = ldv<VEC>(p.gout + ro);
        st.c_a[k] = __ldg(p.er + rh + L.hk[k]);
        st.c_m[k] = __ldg(p.row_max + rh + L.hk[k]);
        const float sv = __ldg(p.row_sum + rh + L.hk[k]);
        st.c_inv[k] = sv > 0.f ? 1.f / sv : 0.f;
        part = dotv(st.cen[k], ldv<VEC>(p.out + ro));
      }
    }
    if (!SRC_PARALLEL) {                       // every lane of the group takes part in the shuffles
      st.c_dot[k] = head_sum(part, p.lph, L.gmask, GROUP);
      if (write_dot && L.act[k] && L.off[k] % p.dim == 0) p.dot[rh + L.hk[k]] = st.c_dot[k];
    }
  }
}

template <int VEC, int GROUP, int NACC, bool SRC_PARALLEL, class P>
__device__ __forceinline__ void gat_bwd_edges(const P& p, const Lanes<VEC, GROUP, NACC>& L, int beg, int end,
                                              int first_batch, int batch_step, BwdState<VEC, GROUP, NACC>& st,
                                              int nx_c) {
  using T = typename VecT<VEC>::type;
  constexpr int U = UnrollBwd<NACC>::value;
  int base = beg + first_batch * GROUP;
  for (; base < end; base += batch_step * GROUP) {
    const int n = min(GROUP, end - base);
    const int my_c = nx_c;
    {                                             // column indices of the next batch, one batch ahead
      const int nxb = base + batch_step * GROUP + L.gl;
      nx_c = (nxb < end) ? ld_stream(p.col + nxb) : 0;
    }
    auto group = [&](auto uu, int j) {          // exactly-sized groups, see gat_fwd_edges
      constexpr int UU = decltype(uu)::value;
      T nb[UU][NACC];
      float pre[UU][NACC], mm[UU][NACC], inv[UU][NACC], dt[UU][NACC];
#pragma unroll
      for (int u = 0; u < UU; ++u) {
        const int c = __shfl_sync(L.gmask, my_c, j + u, GROUP);
        const size_t ch = static_cast<size_t>(c) * p.heads;
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
          zero_vec(nb[u][k]);
          pre[u][k] = mm[u][k] = inv[u][k] = dt[u][k] = 0.f;
          if (L.act[k]) {
            if (SRC_PARALLEL) {      // neighbour = destination: its er, max, sum, dot, dout row
              nb[u][k] = ldv<VEC>(p.gout + static_cast<size_t>(c) * p.hd + L.off[k]);
              pre[u][k] = st.c_a[k] + __ldg(p.er + ch + L.hk[k]);
              mm[u][k] = __ldg(p.row_max + ch + L.hk[k]);
              const float sv = __ldg(p.row_sum + ch + L.hk[k]);
              inv[u][k] = sv > 0.f ? 1.f / sv : 0.f;
              dt[u][k] = __ldg(p.dot + ch + L.hk[k]);
            } else {                 // neighbour = source: its el and feature row
              nb[u][k] = ldf<VEC>(p.feat + static_cast<size_t>(c) * p.hd + L.off[k]);
              pre[u][k] = __ldg(p.el + ch + L.hk[k]) + st.c_a[k];
              mm[u][k] = st.c_m[k];
              inv[u][k] = st.c_inv[k];
              dt[u][k] = st.c_dot[k];
            }
          }
        }
      }
#pragma unroll
      for (int u = 0; u < UU; ++u) {
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
          const float part = L.act[k] ? dotv(st.cen[k], nb[u][k]) : 0.f;
          const float dalpha = head_sum(part, p.lph, L.gmask, GROUP);      // <dout[v,h,:], feat[u,h,:]>
          if (L.act[k]) {
            const float alpha = __expf(lrelu(pre[u][k], p.slope) - mm[u][k]) * inv[u][k];
            const float g = alpha * (dalpha - dt[u][k]) * (pre[u][k] > 0.f ? 1.f : p.slope);
            st.acch[k] += g;
            if (SRC_PARALLEL) fma_vec(st.accv[k], alpha, nb[u][k]);
          }
        }
      }
    };
    for_exact_groups<U>(n, group);
  }
}

template <int VEC, int GROUP, int NACC, bool SRC_PARALLEL, class P>
__device__ __forceinline__ void gat_bwd_store(const P& p, const Lanes<VEC, GROUP, NACC>& L, int row,
                                              BwdState<VEC, GROUP, NACC>& st) {
  const size_t rh = static_cast<size_t>(row) * p.heads;
#pragma unroll
  for (int k = 0; k < NACC; ++k) {
    if (!L.act[k]) continue;
    if (SRC_PARALLEL) {
      using FT = typename P::feat_t;
      stf<VEC>(reinterpret_cast<FT*>(p.o_vec) + static_cast<size_t>(row) * p.hd + L.off[k], st.accv[k]);
    }
    if (L.off[k] % p.dim == 0) p.o_head[rh + L.hk[k]] = st.acch[k];
  }
}

template <typename FT, int VEC, int GROUP, int NACC, bool SRC_PARALLEL>
__global__ void __launch_bounds__(kGatThreads) gat_bwd_kernel(const GatParams<FT> p) {
  Lanes<VEC, GROUP, NACC> L;
  L.init(p);
  const int warp = blockIdx.x * (kGatThreads / 32) + (threadIdx.x >> 5);
  const int row = warp * (32 / GROUP) + (threadIdx.x & 31) / GROUP;
  if (row < p.num_rows) {
    const int beg = __ldg(p.row_off + row), end = __ldg(p.row_off + row + 1);
    if (!(p.hub_threshold > 0 && (end - beg) > p.hub_threshold)) {
      BwdState<VEC, GROUP, NACC> st;
      gat_bwd_prologue<VEC, GROUP, NACC, SRC_PARALLEL>(p, L, row, st, true);
      gat_bwd_edges<VEC, GROUP, NACC, SRC_PARALLEL>(p, L, beg, end, 0, 1, st, first_cols<GROUP>(p, beg, end, 0, L.gl));
      gat_bwd_store<VEC, GROUP, NACC, SRC_PARALLEL>(p, L, row, st);
    }
  }
  grid_dependency_wait();
}


// Hub rows (longer than the view's hub threshold) in two tiers, for all three passes (KIND as above):
//   * a row of up to kGatGiantEdges edges is walked by ONE CTA: its 8 warps take strided batches and merge their
//     partials (forward: online-softmax states (max, sum, acc); backward: plain sums) through shuffles and
//     shared memory;
//   * a longer row is walked by a whole thread-block cluster (8 CTAs, 64 warps) and the leader CTA merges the
//     CTA partials over distributed shared memory -- one CTA needs ~100 us of dependent L2 round trips for the
//     8.5 K-edge rows of config 3, which used to be the critical path of every pass.
// Every merge runs in a fixed order: deterministic, no atomics, no scratch in HBM.  Entry i of the hub list
// is tested by cluster i % n_clusters (giant?) and by CTA i % n_ctas (not giant?), so the list may be in any
// order; StaticGraph sorts it by length so that the giant rows start first, one per cluster.
constexpr int kGatCluster = 8;
constexpr int kGatGiantEdges = 1024;

template <int NACC> struct HubThreads { static constexpr int value = NACC >= 4 ? kGatHubThreads / 2 : kGatHubThreads; };

template <typename FT, int VEC, int GROUP, int NACC, int KIND>
__global__ void __cluster_dims__(kGatCluster, 1, 1) __launch_bounds__(HubThreads<NACC>::value, NACC == 1 ? 4 : 1)
    gat_hub_kernel(const GatParams<FT> p) {
  using T = typename VecT<VEC>::type;
  namespace cg = cooperative_groups;
  constexpr int WARPS = HubThreads<NACC>::value / 32;
  constexpr int GPW = 32 / GROUP;
  constexpr bool FWD = KIND == 0;
  constexpr bool SRC = KIND == 2;
  __shared__ T s_v[WARPS][GROUP * NACC];
  __shared__ float s_a[WARPS][GROUP * NACC], s_b[FWD ? WARPS : 1][GROUP * NACC];
  __shared__ T c_v[GROUP * NACC];                       // this CTA's partial, read by the cluster leader
  __shared__ float c_a[GROUP * NACC], c_b[GROUP * NACC];
  // the row kernel is launched behind this one as a programmatic dependent: the two write disjoint rows
  asm volatile("griddepcontrol.launch_dependents;");
  cg::cluster_group cluster = cg::this_cluster();
  Lanes<VEC, GROUP, NACC> L;
  L.init(p);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int crank = static_cast<int>(cluster.block_rank());
  const int n_hub = min(__ldg(p.hub_count), p.hub_capacity);
  const bool leader_lanes = wid == 0 && lane < GROUP;

  // Walk edges [beg,end) of `row` with `slots` cooperating (warp, group) slots, this thread's being `slot`; merge the
  // CTA's partials into warp 0, lanes [0, GROUP) (registers `st`) in a fixed order.
  using State = typename std::conditional<FWD, FwdState<VEC, GROUP, NACC>, BwdState<VEC, GROUP, NACC>>::type;
  State st;
  auto cta_partial = [&](int row, int beg, int end, int slot, int slots, bool write_dot) {
    const int c_first = first_cols<GROUP>(p, beg, end, slot, L.gl);
    if constexpr (FWD) {
      st.init();
      gat_fwd_edges<VEC, GROUP, NACC>(p, L, row, beg, end, slot, slots, st, c_first);
#pragma unroll
      for (int o = GROUP; o < 32; o <<= 1) {            // groups of one warp -> lanes [0, GROUP)
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
          const float m2 = __shfl_xor_sync(0xffffffffu, st.m[k], o);
          const float s2 = __shfl_xor_sync(0xffffffffu, st.s[k], o);
          const T a2 = shfl_xor_t(0xffffffffu, st.acc[k], o);
          st.merge(k, m2, s2, a2);
        }
      }
      if (lane < GROUP) {
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
          s_v[wid][k * GROUP + lane] = st.acc[k];
          s_a[wid][k * GROUP + lane] = st.m[k];
          s_b[wid][k * GROUP + lane] = st.s[k];
        }
      }
      __syncthreads();
      if (leader_lanes) {
#pragma unroll
        for (int k = 0; k < NACC; ++k)
          for (int w = 1; w < WARPS; ++w)
            st.merge(k, s_a[w][k * GROUP + lane], s_b[w][k * GROUP + lane], s_v[w][k * GROUP + lane]);
      }
    } else {
      gat_bwd_prologue<VEC, GROUP, NACC, SRC>(p, L, row, st, write_dot && leader_lanes);
      gat_bwd_edges<VEC, GROUP, NACC, SRC>(p, L, beg, end, slot, slots, st, c_first);
#pragma unroll
      for (int o = GROUP; o < 32; o <<= 1) {
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
          st.acch[k] += __shfl_xor_sync(0xffffffffu, st.acch[k], o);
          add_vec(st.accv[k], shfl_xor_t(0xffffffffu, st.accv[k], o));
        }
      }
      if (lane < GROUP) {
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
          s_v[wid][k * GROUP + lane] = st.accv[k];
          s_a[wid][k * GROUP + lane] = st.acch[k];
        }
      }
      __syncthreads();
      if (leader_lanes) {
#pragma unroll
        for (int k = 0; k < NACC; ++k)
          for (int w = 1; w < WARPS; ++w) {
            add_vec(st.accv[k], s_v[w][k * GROUP + lane]);
            st.acch[k] += s_a[w][k * GROUP + lane];
          }
      }
    }
  };
  auto store_row = [&](int row, bool nonempty) {         // warp 0, lanes [0, GROUP)
    if constexpr (FWD) gat_fwd_store<VEC, GROUP, NACC>(p, L, row, nonempty, st);
    else gat_bwd_store<VEC, GROUP, NACC, SRC>(p, L, row, st);
  };

  // tier 2: giant rows, one per cluster at a time (the same decisions in every CTA of the cluster)
  const int cluster_id = blockIdx.x / kGatCluster, n_clusters = gridDim.x / kGatCluster;
  for (int i = cluster_id; i < n_hub; i += n_clusters) {
    const int row = __ldg(p.hub_rows + i);
    const int beg = __ldg(p.row_off + row), end = __ldg(p.row_off + row + 1);
    if ((end - beg) <= kGatGiantEdges) continue;
    cta_partial(row, beg, end, (crank * WARPS + wid) * GPW + lane / GROUP, kGatCluster * WARPS * GPW, crank == 0);
    if (leader_lanes) {
#pragma unroll
      for (int k = 0; k < NACC; ++k) {
        if constexpr (FWD) {
          c_v[k * GROUP + lane] = st.acc[k];
          c_a[k * GROUP + lane] = st.m[k];
          c_b[k * GROUP + lane] = st.s[k];
        } else {
          c_v[k * GROUP + lane] = st.accv[k];
          c_a[k * GROUP + lane] = st.acch[k];
        }
      }
    }
    cluster.sync();                                      // every CTA's partial is in its c_* arrays
    if (crank == 0 && leader_lanes) {                    // CTAs of the cluster, fixed order, over DSMEM
      for (int c = 1; c < kGatCluster; ++c) {
        const T* rv = cluster.map_shared_rank(c_v, c);
        const float* ra = cluster.map_shared_rank(c_a, c);
        const float* rb = cluster.map_shared_rank(c_b, c);
#pragma unroll
        for (int k = 0; k < NACC; ++k) {
          if constexpr (FWD) {
            st.merge(k, ra[k * GROUP + lane], rb[k * GROUP + lane], rv[k * GROUP + lane]);
          } else {
            add_vec(st.accv[k], rv[k * GROUP + lane]);
            st.acch[k] += ra[k * GROUP + lane];
          }
        }
      }
      store_row(row, true);
    }
    cluster.sync();                                      // peers keep c_* alive until the leader has read them
  }
  // tier 1: the other hub rows, one per CTA at a time
  for (int i = blockIdx.x; i < n_hub; i += gridDim.x) {
    const int row = __ldg(p.hub_rows + i);
    const int beg = __ldg(p.row_off + row), end = __ldg(p.row_off + row + 1);
    if ((end - beg) > kGatGiantEdges) continue;
    cta_partial(row, beg, end, wid * GPW + lane / GROUP, WARPS * GPW, true);
    if (leader_lanes) store_row(row, end > beg);
    __syncthreads();                                     // s_* are rewritten by the next row
  }
}

// Row-queue form of the three row kernels for one row per warp (GROUP = 32).  On a power-law graph most rows
// hold a handful of edges, so a one-row-per-warp grid is a string of dependent L2 round trips per block
// (row_offset -> column -> neighbour rows -> store) plus one block launch per 8 rows.  Here a block owns
// rows_per_block consecutive rows, its warps draw rows from a shared-memory counter, and the row_offset pair of
// the row after next and the first column batch of the next row are in flight while a row is processed.
// KIND: 0 forward, 1 backward pass A (destination-parallel), 2 backward pass B (source-parallel).
constexpr int kGatRowsPerWarp = 16;

// GQ: global row queue as in agg.cu (persistent grid, warps draw chunks of rows_per_block rows from the view's device
// counter; the last block rearms it): config 3 has 1323 blocks of 128 rows on 592 block slots, i.e. 2.2 waves whose
// last one is a third full -- with the queue every warp stays busy until the rows run out.
template <typename FT, int VEC, int NACC, int KIND, bool GQ = false>
__global__ void __launch_bounds__(kGatThreads, NACC == 1 ? 4 : 1) gat_rows_pipe_kernel(const GatParams<FT> p, int rows_per_block) {
  constexpr int GROUP = 32;
  __shared__ int next_row;
  Lanes<VEC, GROUP, NACC> L;
  L.init(p);
  const int lane = threadIdx.x & 31;
  const int first = GQ ? 0 : blockIdx.x * rows_per_block;
  const int last = GQ ? p.num_rows : min(first + rows_per_block, p.num_rows);
  int q_cur = 0, q_pos = rows_per_block, q_nxt = 0;
  if constexpr (GQ) {
    if (lane == 0) q_nxt = atomicAdd(p.queue, 1);
  } else {
    if (threadIdx.x == 0) next_row = first;
    __syncthreads();
  }
  auto draw = [&]() {
    if constexpr (GQ) {
      if (q_pos == rows_per_block && q_cur < p.num_rows) {
        q_cur = __shfl_sync(0xffffffffu, q_nxt, 0) * rows_per_block;
        q_pos = 0;
        if (lane == 0 && q_cur < p.num_rows) q_nxt = atomicAdd(p.queue, 1);
      }
      return q_cur + q_pos++;
    } else {
      int r = 0;
      if (lane == 0) r = atomicAdd(&next_row, 1);
      return __shfl_sync(0xffffffffu, r, 0);
    }
  };
  auto finish = [&]() {
    if constexpr (GQ) {
      __syncthreads();
      if (threadIdx.x == 0 && atomicAdd(p.queue + 1, 1) == static_cast<int>(gridDim.x) - 1) {
        p.queue[0] = 0;
        p.queue[1] = 0;
        __threadfence();
      }
    }
    grid_dependency_wait();
  };
  auto offsets = [&](int row, int& beg, int& end) {      // end = -1: nothing to do (past the end)
    beg = 0;
    end = -1;
    if (row < last) {
      beg = __ldg(p.row_off + row);
      end = __ldg(p.row_off + row + 1);
    }
  };
  auto drop_hub = [&](int& beg, int& end) {              // hub rows belong to the block-per-row kernel
    if (p.hub_threshold > 0 && (end - beg) > p.hub_threshold) beg = 0, end = -1;
  };
  int row0 = draw();
  if (row0 >= last) {
    finish();
    return;
  }
  int beg0, end0, beg1, end1;
  offsets(row0, beg0, end0);
  int row1 = draw();
  offsets(row1, beg1, end1);
  drop_hub(beg0, end0);
  int c0 = first_cols<GROUP>(p, beg0, end0, 0, lane);
  while (row0 < last) {
    const int row2 = draw();
    int beg2, end2;
    offsets(row2, beg2, end2);
    drop_hub(beg1, end1);
    const int c1 = first_cols<GROUP>(p, beg1, end1, 0, lane);
    if (end0 >= 0) {
      if constexpr (KIND == 0) {
        FwdState<VEC, GROUP, NACC> st;
        st.init();
        gat_fwd_edges<VEC, GROUP, NACC>(p, L, row0, beg0, end0, 0, 1, st, c0);
        gat_fwd_store<VEC, GROUP, NACC>(p, L, row0, end0 > beg0, st);
      } else {
        BwdState<VEC, GROUP, NACC> st;
        gat_bwd_prologue<VEC, GROUP, NACC, KIND == 2>(p, L, row0, st, true);
        gat_bwd_edges<VEC, GROUP, NACC, KIND == 2>(p, L, beg0, end0, 0, 1, st, c0);
        gat_bwd_store<VEC, GROUP, NACC, KIND == 2>(p, L, row0, st);
      }
    }
    row0 = row1; beg0 = beg1; end0 = end1; c0 = c1;
    row1 = row2; beg1 = beg2; end1 = end2;
  }
  finish();
}

// Rows a warp draws from the global queue at a time (STG_GAT_CHUNK; 0 = static block ranges; read once).
inline int gat_queue_chunk() {
  static const int v = [] {
    const char* e = getenv("STG_GAT_CHUNK");
    const int c = e ? atoi(e) : 2;      // config 3, fwd / bwd kernels: static 0.245 / 0.686 ms, chunk 4: 0.250 / 0.637, chunk 2: 0.245 / 0.623
    return c < 0 ? 0 : (c > 1024 ? 1024 : c);
  }();
  return v;
}

// Hub CTAs per SM (STG_GAT_HUB_GRID; read once): four fill the register file until they exit, fewer leave room for the
// row kernel from the start but serve fewer hub rows at a time.
inline int gat_hub_grid_mult() {
  static const int v = [] {
    const char* e = getenv("STG_GAT_HUB_GRID");
    const int c = e ? atoi(e) : 4;
    return c < 1 ? 1 : (c > 8 ? 8 : c);
  }();
  return v;
}

template <typename FT, int VEC, int GROUP, int NACC>
int launch_gat(const GatParams<FT>& p, int which, cudaStream_t s) {
  const int rows_per_block = (kGatThreads / 32) * (32 / GROUP);
  const int blocks = (p.num_rows + rows_per_block - 1) / rows_per_block;
  if (blocks <= 0) return STG_OK;
  const bool hubs = p.hub_threshold > 0 && p.hub_rows != nullptr;
  const int hub_grid = gat_hub_grid_mult() * (sm_count() / kGatCluster) * kGatCluster;   // 8-warp CTAs of <= 64 registers per SM
  // Hub rows first: the longest rows are the critical path, the row kernel fills the SMs they leave idle.
  if (hubs) {
    constexpr int ht = HubThreads<NACC>::value;
    if (which == 0) gat_hub_kernel<FT, VEC, GROUP, NACC, 0><<<hub_grid, ht, 0, s>>>(p);
    else if (which == 1) gat_hub_kernel<FT, VEC, GROUP, NACC, 1><<<hub_grid, ht, 0, s>>>(p);
    else gat_hub_kernel<FT, VEC, GROUP, NACC, 2><<<hub_grid, ht, 0, s>>>(p);
    STG_LAUNCH_CHECK("gat hub kernel");
  }
  if constexpr (GROUP == 32) {
    if (p.num_rows >= 4096) {      // the queue pays off once there are several blocks per SM
      if (p.queue != nullptr && gat_queue_chunk() > 0) {
        const int gblocks = std::min(sm_count() * (NACC == 1 ? 4 : 1), (p.num_rows + 7) / 8);
        const int ch = gat_queue_chunk();
        if (which == 0) STG_CUDA(launch_overlapped(gat_rows_pipe_kernel<FT, VEC, NACC, 0, true>, gblocks, kGatThreads, s, hubs, p, ch));
        else if (which == 1) STG_CUDA(launch_overlapped(gat_rows_pipe_kernel<FT, VEC, NACC, 1, true>, gblocks, kGatThreads, s, hubs, p, ch));
        else STG_CUDA(launch_overlapped(gat_rows_pipe_kernel<FT, VEC, NACC, 2, true>, gblocks, kGatThreads, s, hubs, p, ch));
        STG_LAUNCH_CHECK("gat rows (global queue) kernel");
        return STG_OK;
      }
      const int rpb = (kGatThreads / 32) * kGatRowsPerWarp;
      const int pblocks = (p.num_rows + rpb - 1) / rpb;
      if (which == 0) STG_CUDA(launch_overlapped(gat_rows_pipe_kernel<FT, VEC, NACC, 0>, pblocks, kGatThreads, s, hubs, p, rpb));
      else if (which == 1) STG_CUDA(launch_overlapped(gat_rows_pipe_kernel<FT, VEC, NACC, 1>, pblocks, kGatThreads, s, hubs, p, rpb));
      else STG_CUDA(launch_overlapped(gat_rows_pipe_kernel<FT, VEC, NACC, 2>, pblocks, kGatThreads, s, hubs, p, rpb));
      STG_LAUNCH_CHECK("gat rows (queue) kernel");
      return STG_OK;
    }
  }
  if (which == 0) gat_fwd_kernel<FT, VEC, GROUP, NACC><<<blocks, kGatThreads, 0, s>>>(p);
  else if (which == 1) gat_bwd_kernel<FT, VEC, GROUP, NACC, false><<<blocks, kGatThreads, 0, s>>>(p);
  else gat_bwd_kernel<FT, VEC, GROUP, NACC, true><<<blocks, kGatThreads, 0, s>>>(p);
  STG_LAUNCH_CHECK("gat kernel");
  return STG_OK;
}

template <typename FT, int VEC>
int dispatch_gat(const GatParams<FT>& p, int which, cudaStream_t s) {
  const int nvec = p.hd / VEC;
  if (nvec <= 1) return launch_gat<FT, VEC, 1, 1>(p, which, s);
  if (nvec <= 2) return launch_gat<FT, VEC, 2, 1>(p, which, s);
  if (nvec <= 4) return launch_gat<FT, VEC, 4, 1>(p, which, s);
  if (nvec <= 8) return launch_gat<FT, VEC, 8, 1>(p, which, s);
  if (nvec <= 16) return launch_gat<FT, VEC, 16, 1>(p, which, s);
  if (nvec <= 32) return launch_gat<FT, VEC, 32, 1>(p, which, s);
  if (nvec <= 64) return launch_gat<FT, VEC, 32, 2>(p, which, s);
  if (nvec <= 128) return launch_gat<FT, VEC, 32, 4>(p, which, s);
  set_error("heads*dim = %d is wider than the fused GAT kernels support (512 floats with dim %% 4 == 0)", p.hd);
  return STG_ERR_UNSUPPORTED;
}

template <typename FT>
int run_gat(GatParams<FT> p, int which, bool aligned, cudaStream_t s) {
  const int vec = (p.dim % 4 == 0 && aligned) ? 4 : 1;
  p.lph = p.dim / vec;
  if ((p.lph & (p.lph - 1)) != 0 || p.lph > 32) {
    set_error("fused GAT kernels need dim/%d = %d lanes per head to be a power of two <= 32 (dim = %d)", vec, p.lph,
              p.dim);
    return STG_ERR_UNSUPPORTED;
  }
  return vec == 4 ? dispatch_gat<FT, 4>(p, which, s) : dispatch_gat<FT, 1>(p, which, s);
}

int check_view(const StgCsrView* g) {
  STG_CHECK_ARG(g && g->row_offset, "graph view / row_offset is NULL");
  STG_CHECK_ARG(g->num_edges == 0 || g->column_indices, "column_indices is NULL");
  return STG_OK;
}

template <typename FT>
void bind_view(GatParams<FT>& p, const StgCsrView* g) {
  p.row_off = g->row_offset;
  p.col = g->column_indices;
  p.queue = g->work_queue;
  const bool hubs = g->hub_rows && g->hub_count && g->hub_threshold > 0;
  p.hub_rows = hubs ? g->hub_rows : nullptr;
  p.hub_count = hubs ? g->hub_count : nullptr;
  p.hub_threshold = hubs ? g->hub_threshold : 0;
  p.hub_capacity = hubs ? g->hub_capacity : 0;
}

// VEC = 4 needs four consecutive feat / d_feat elements to be one aligned access (16 bytes of fp32, 8 of 16-bit rows)
template <typename FT>
bool vec4_aligned(const void* p) {
  return (reinterpret_cast<uintptr_t>(p) & (4 * sizeof(FT) - 1)) == 0;
}

template <typename FT>
int gat_fwd(const StgCsrView* g_in, const float* el, const float* er, const FT* feat, int32_t heads, int32_t dim,
            float slope, float* out, float* row_max, float* row_sum, void* stream) {
  int rc = check_view(g_in);
  if (rc != STG_OK) return rc;
  STG_CHECK_ARG(heads > 0 && dim > 0, "heads and dim must be positive");
  if (g_in->num_nodes == 0) return STG_OK;
  STG_CHECK_ARG(el && er && feat && out && row_max && row_sum, "NULL tensor");
  GatParams<FT> p{};
  bind_view(p, g_in);
  p.num_rows = g_in->num_nodes;
  p.heads = heads;
  p.dim = dim;
  p.hd = heads * dim;
  p.slope = slope;
  p.el = el;
  p.er = er;
  p.feat = feat;
  p.row_max = row_max;
  p.row_sum = row_sum;
  p.o_vec = out;
  return run_gat(p, 0, vec4_aligned<FT>(feat) && aligned16(out), as_stream(stream));
}

template <typename FT>
int gat_bwd(const StgCsrView* g_in, const StgCsrView* g_out, const float* el, const float* er, const FT* feat,
            const float* out, const float* grad_out, const float* row_max, const float* row_sum, int32_t heads,
            int32_t dim, float slope, FT* d_feat, float* d_el, float* d_er, float* dot_scratch, void* stream) {
  int rc = check_view(g_in);
  if (rc != STG_OK) return rc;
  rc = check_view(g_out);
  if (rc != STG_OK) return rc;
  STG_CHECK_ARG(heads > 0 && dim > 0, "heads and dim must be positive");
  STG_CHECK_ARG(g_in->num_nodes == g_out->num_nodes, "forward / backward views disagree on the node count");
  if (g_in->num_nodes == 0) return STG_OK;
  STG_CHECK_ARG(el && er && feat && out && grad_out && row_max && row_sum && d_feat && d_el && d_er && dot_scratch,
                "NULL tensor");
  GatParams<FT> p{};
  p.num_rows = g_in->num_nodes;
  p.heads = heads;
  p.dim = dim;
  p.hd = heads * dim;
  p.slope = slope;
  p.el = el;
  p.er = er;
  p.feat = feat;
  p.out = out;
  p.gout = grad_out;
  p.row_max = const_cast<float*>(row_max);
  p.row_sum = const_cast<float*>(row_sum);
  p.dot = dot_scratch;
  const bool al = vec4_aligned<FT>(feat) && aligned16(out) && aligned16(grad_out) && vec4_aligned<FT>(d_feat);
  cudaStream_t s = as_stream(stream);
  // pass A: destination-parallel on the in-edge view -> dot, d_er
  bind_view(p, g_in);
  p.o_vec = nullptr;
  p.o_head = d_er;
  rc = run_gat(p, 1, al, s);
  if (rc != STG_OK) return rc;
  // pass B: source-parallel on the out-edge view -> d_feat, d_el
  bind_view(p, g_out);
  p.o_vec = reinterpret_cast<float*>(d_feat);
  p.o_head = d_el;
  return run_gat(p, 2, al, s);
}

int check_dtype(int32_t dtype) {
  STG_CHECK_ARG(dtype == STG_DTYPE_BF16 || dtype == STG_DTYPE_F16, "unknown dtype code %d (STG_DTYPE_BF16 = 1, STG_DTYPE_F16 = 2)",
                dtype);
  return STG_OK;
}

}  // namespace
}  // namespace stg

using namespace stg;

STG_API int stg_gat_softmax_fwd_f32(const StgCsrView* g_in, const float* el, const float* er, const float* feat,
                                    int32_t heads, int32_t dim, float slope, float* out, float* row_max,
                                    float* row_sum, void* stream) {
  return gat_fwd(g_in, el, er, feat, heads, dim, slope, out, row_max, row_sum, stream);
}

STG_API int stg_gat_softmax_bwd_f32(const StgCsrView* g_in, const StgCsrView* g_out, const float* el, const float* er,
                                    const float* feat, const float* out, const float* grad_out, const float* row_max,
                                    const float* row_sum, int32_t heads, int32_t dim, float slope, float* d_feat,
                                    float* d_el, float* d_er, float* dot_scratch, void* stream) {
  return gat_bwd(g_in, g_out, el, er, feat, out, grad_out, row_max, row_sum, heads, dim, slope, d_feat, d_el, d_er,
                 dot_scratch, stream);
}

STG_API int stg_gat_softmax_fwd_h16(const StgCsrView* g_in, const float* el, const float* er, const void* feat,
                                    int32_t heads, int32_t dim, int32_t dtype, float slope, float* out, float* row_max,
                                    float* row_sum, void* stream) {
  const int rc = check_dtype(dtype);
  if (rc != STG_OK) return rc;
  if (dtype == STG_DTYPE_BF16)
    return gat_fwd(g_in, el, er, static_cast<const __nv_bfloat16*>(feat), heads, dim, slope, out, row_max, row_sum, stream);
  return gat_fwd(g_in, el, er, static_cast<const __half*>(feat), heads, dim, slope, out, row_max, row_sum, stream);
}

STG_API int stg_gat_softmax_bwd_h16(const StgCsrView* g_in, const StgCsrView* g_out, const float* el, const float* er,
                                    const void* feat, const float* out, const float* grad_out, const float* row_max,
                                    const float* row_sum, int32_t heads, int32_t dim, int32_t dtype, float slope,
                                    void* d_feat, float* d_el, float* d_er, float* dot_scratch, void* stream) {
  const int rc = check_dtype(dtype);
  if (rc != STG_OK) return rc;
  if (dtype == STG_DTYPE_BF16)
    return gat_bwd(g_in, g_out, el, er, static_cast<const __nv_bfloat16*>(feat), out, grad_out, row_max, row_sum, heads,
                   dim, slope, static_cast<__nv_bfloat16*>(d_feat), d_el, d_er, dot_scratch, stream);
  return gat_bwd(g_in, g_out, el, er, static_cast<const __half*>(feat), out, grad_out, row_max, row_sum, heads, dim,
                 slope, static_cast<__half*>(d_feat), d_el, d_er, dot_scratch, stream);
}
