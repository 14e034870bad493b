// Neighbour aggregation over 16-bit feature rows (bf16 or fp16) with fp32 accumulation, for sm_100a.
//
//   out[r,:] = row_scale[r] * sum_{e in row r} nbr_scale[col[e]] * edge_scale[eid(e)] * x[col[e],:]
//
// x and out are [N, F] row-major in the same 16-bit type; the scales and the packed {col, scale} records stay fp32.
// Every product and the running sum are fp32, and the row is rounded to the 16-bit type once, when it is stored.
// This is what the GCN aggregation computes under torch.autocast: the gathered row is half as many bytes as in the
// fp32 kernels of agg.cu (200 instead of 400 bytes per edge at F = 100), the rest of the per-edge work is the same.
//
// Shape (a simpler form of agg.cu's, assign mode only):
//   * one row per warp; lane L owns VEC (8/4/2/1) consecutive elements x NACC (1/2/4) chunks of 32 * VEC, loaded
//     with the widest access alignment allows (16/8/4/2 bytes); wider rows are walked in column chunks;
//   * the {column, scale} of the next 32 edges are loaded one per lane, a batch ahead, and broadcast by shuffles;
//   * large graphs whose view carries a global row queue: a persistent grid whose warps draw chunks of rows from
//     StgCsrView::work_queue with agg.cu's protocol (the last block rearms {0, 0}), with the row offsets and the first
//     edge batch of the next rows in flight while a row is summed; otherwise one row per warp, static;
//   * rows longer than hub_threshold (when the view has a hub list) are summed by one 512-thread CTA each, warps
//     taking interleaved edge batches and reduced through shared memory in warp order.
// Each row is summed in one fixed order whatever the schedule: deterministic, no atomics on data.
#include "common.cuh"

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <type_traits>

namespace stg {
namespace {

constexpr int kH16Threads = 256;
constexpr int kH16HubThreads = 512;
constexpr int kH16QueueChunk = 4;   // rows a warp draws from the global queue at a time (agg.cu's default)

enum H16Mode { kH16Plain = 0, kH16Packed = 1 };

template <typename T> struct H16;
template <> struct H16<__nv_bfloat16> {   // (widened by unpack's shift)
  using T2 = __nv_bfloat162;
  static __device__ __forceinline__ T2 from_f2(float a, float b) { return __floats2bfloat162_rn(a, b); }
  static __device__ __forceinline__ __nv_bfloat16 from_f(float a) { return __float2bfloat16_rn(a); }
};
template <> struct H16<__half> {
  using T2 = __half2;
  static __device__ __forceinline__ float2 to_f2(T2 v) { return __half22float2(v); }
  static __device__ __forceinline__ T2 from_f2(float a, float b) { return __floats2half2_rn(a, b); }
  static __device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
  static __device__ __forceinline__ __half from_f(float a) { return __float2half_rn(a); }
};

// One lane's access: VEC 16-bit elements.
template <int VEC> struct Raw;
template <> struct Raw<8> { using type = uint4; };
template <> struct Raw<4> { using type = uint2; };
template <> struct Raw<2> { using type = unsigned int; };
template <> struct Raw<1> { using type = unsigned short; };

template <typename T, int VEC>
__device__ __forceinline__ void unpack(const typename Raw<VEC>::type& r, float (&f)[VEC]) {
  if constexpr (std::is_same_v<T, __nv_bfloat16>) {
    // bf16 -> fp32 is a 16-bit shift: one integer op per element.  The cuda_bf16.h pair conversion compiles to ~1.7 per
    // element on sm_100a, and with it the issue-bound config-5 row kernel took 2.26 ms against 1.85 ms for fp16.
    if constexpr (VEC == 1) {
      f[0] = __uint_as_float(static_cast<unsigned>(r) << 16);
    } else {
      const unsigned* w = reinterpret_cast<const unsigned*>(&r);
#pragma unroll
      for (int i = 0; i < VEC / 2; ++i) {
        f[2 * i] = __uint_as_float(w[i] << 16);
        f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
      }
    }
  } else if constexpr (VEC == 1) {
    f[0] = H16<T>::to_f(*reinterpret_cast<const T*>(&r));
  } else {
    const auto* h = reinterpret_cast<const typename H16<T>::T2*>(&r);
#pragma unroll
    for (int i = 0; i < VEC / 2; ++i) {
      const float2 v = H16<T>::to_f2(h[i]);
      f[2 * i] = v.x;
      f[2 * i + 1] = v.y;
    }
  }
}

template <typename T, int VEC>
__device__ __forceinline__ typename Raw<VEC>::type pack(const float (&f)[VEC]) {
  typename Raw<VEC>::type r;
  if constexpr (VEC == 1) {
    *reinterpret_cast<T*>(&r) = H16<T>::from_f(f[0]);
  } else {
    auto* h = reinterpret_cast<typename H16<T>::T2*>(&r);
#pragma unroll
    for (int i = 0; i < VEC / 2; ++i) h[i] = H16<T>::from_f2(f[2 * i], f[2 * i + 1]);
  }
  return r;
}

template <typename T>
struct H16Params {
  const int32_t* __restrict__ row_off;
  const int32_t* __restrict__ col;
  const int32_t* __restrict__ eids;
  const int32_t* __restrict__ hub_rows;
  const int32_t* __restrict__ hub_count;
  const int2* __restrict__ meta;   // kH16Packed: {column, scale bits} per CSR slot (stg_csr_pack_edge_meta_f32)
  int* queue;                      // StgCsrView::work_queue or NULL
  int num_rows;
  int eid_base;
  int eids_identity;
  int hub_threshold;               // 0: no hub split
  int hub_capacity;
  const T* __restrict__ x;         // offset to the chunk's first column
  T* __restrict__ out;             // same
  int ld;                          // elements between consecutive rows of x and of out (= feat)
  int width;                       // elements of this chunk
  const float* __restrict__ ns;
  const float* __restrict__ es;
  const float* __restrict__ rs;
};

// Column and combined scale of edge e (0 / 0.f past the end of its row).  The plain product order is that of
// pack_edge_meta_kernel, so plain and packed sums agree bit for bit.
template <int MODE, typename P>
__device__ __forceinline__ void edge_record(const P& p, int e, int end, int& c, float& s) {
  c = 0;
  s = 0.f;
  if (e >= end) return;
  if constexpr (MODE == kH16Packed) {
    const int2 m = __ldcs(p.meta + e);
    c = m.x;
    s = __int_as_float(m.y);
  } else {
    c = ld_stream(p.col + e);
    float sc = 1.f;
    if (p.ns) sc = __ldg(p.ns + c);
    if (p.es) {
      const int eid = p.eids_identity ? e : (ld_stream(p.eids + e) - p.eid_base);
      sc *= __ldg(p.es + eid);
    }
    s = sc;
  }
}

// acc += sum over the edges of [beg, end) in batches of 32 starting at beg + 32 * first, every `step`-th batch.
// (c, s): this lane's record of the first batch, loaded by the caller.  All 32 lanes of the warp take part.
template <typename T, int VEC, int NACC, int MODE>
__device__ __forceinline__ void sum_edges(const H16Params<T>& p, int beg, int end, int first, int step, int lane,
                                          float (&acc)[NACC][VEC], int c, float s) {
  using R = typename Raw<VEC>::type;
  constexpr int UNROLL = NACC == 1 ? 8 : (NACC == 2 ? 4 : 2);
  const char* base[NACC];
  bool live[NACC];
#pragma unroll
  for (int k = 0; k < NACC; ++k) {
    const int o = (lane + 32 * k) * VEC;
    live[k] = o < p.width;
    base[k] = reinterpret_cast<const char*>(p.x + (live[k] ? o : 0));
  }
  const size_t ld_bytes = static_cast<size_t>(p.ld) * sizeof(T);
  auto load = [&](int cc, int k) {
    R v;
    if (live[k]) v = __ldg(reinterpret_cast<const R*>(base[k] + static_cast<size_t>(static_cast<unsigned>(cc)) * ld_bytes));
    else v = R{};
    return v;
  };
  auto fma_row = [&](float sc, const R (&v)[NACC]) {
#pragma unroll
    for (int k = 0; k < NACC; ++k) {
      float f[VEC];
      unpack<T, VEC>(v[k], f);
#pragma unroll
      for (int i = 0; i < VEC; ++i) acc[k][i] = fmaf(sc, f[i], acc[k][i]);
    }
  };
  for (int b = beg + 32 * first; b < end; b += 32 * step) {
    int nc;
    float nsc;
    edge_record<MODE>(p, b + 32 * step + lane, end, nc, nsc);   // next batch in flight
    const int n = min(32, end - b);
    int j = 0;
    for (; j + UNROLL <= n; j += UNROLL) {
      int cc[UNROLL];
      float sc[UNROLL];
      R v[UNROLL][NACC];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        cc[u] = __shfl_sync(0xffffffffu, c, j + u);
        sc[u] = __shfl_sync(0xffffffffu, s, j + u);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
#pragma unroll
        for (int k = 0; k < NACC; ++k) v[u][k] = load(cc[u], k);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) fma_row(sc[u], v[u]);
    }
    if (j < n) {                      // partial group: edges past the row read nothing (x may hold NaN elsewhere)
      int cc[UNROLL];
      float sc[UNROLL];
      R v[UNROLL][NACC];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        cc[u] = __shfl_sync(0xffffffffu, c, (j + u) & 31);
        sc[u] = __shfl_sync(0xffffffffu, s, (j + u) & 31);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
#pragma unroll
        for (int k = 0; k < NACC; ++k) v[u][k] = (j + u < n) ? load(cc[u], k) : R{};
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) fma_row(sc[u], v[u]);
    }
    c = nc;
    s = nsc;
  }
}

template <typename T, int VEC, int NACC>
__device__ __forceinline__ void store_row(const H16Params<T>& p, int row, int lane, float r, float (&acc)[NACC][VEC]) {
  using R = typename Raw<VEC>::type;
  T* dst = p.out + static_cast<size_t>(row) * p.ld;
#pragma unroll
  for (int k = 0; k < NACC; ++k) {
    const int o = (lane + 32 * k) * VEC;
    if (o < p.width) {
      float f[VEC];
#pragma unroll
      for (int i = 0; i < VEC; ++i) f[i] = acc[k][i] * r;
      __stcs(reinterpret_cast<R*>(dst + o), pack<T, VEC>(f));
    }
  }
}

// One row per warp.  GQ: warps of a persistent grid draw chunks of kH16QueueChunk rows from p.queue[0] (the next
// chunk id is fetched while the current chunk is summed) and the last block rearms the queue; otherwise warp w
// takes rows w, w + (all warps), ...  Row offsets are fetched two rows ahead and the first edge batch one row ahead.
template <typename T, int VEC, int NACC, int MODE, bool GQ>
__device__ __forceinline__ void rows_body(const H16Params<T>& p) {
  const int lane = threadIdx.x & 31;
  const int warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  int q_cur = 0, q_pos = kH16QueueChunk, q_nxt = 0, seq = 0;
  if constexpr (GQ) {
    if (lane == 0) q_nxt = atomicAdd(p.queue, 1);
  }
  auto draw = [&]() -> int {                  // next row of this warp, or num_rows when there is none
    if constexpr (GQ) {
      if (q_pos == kH16QueueChunk && q_cur < p.num_rows) {     // warp-uniform
        q_cur = __shfl_sync(0xffffffffu, q_nxt, 0) * kH16QueueChunk;
        q_pos = 0;
        if (lane == 0 && q_cur < p.num_rows) q_nxt = atomicAdd(p.queue, 1);
      }
      const int r = q_cur + q_pos++;
      return r < p.num_rows ? r : p.num_rows;
    } else {
      const long long r = warp + static_cast<long long>(seq++) * nwarps;
      return r < p.num_rows ? static_cast<int>(r) : p.num_rows;
    }
  };
  auto bounds = [&](int row, int& beg, int& end) {   // end = -1: nothing to do (past the end, hub row)
    beg = 0;
    end = -1;
    if (row >= p.num_rows) return;
    beg = __ldg(p.row_off + row);
    end = __ldg(p.row_off + row + 1);
    if (p.hub_threshold > 0 && end - beg > p.hub_threshold) beg = 0, end = -1;
  };

  int row0 = draw(), beg0, end0;
  bounds(row0, beg0, end0);
  int row1 = draw(), beg1, end1;
  bounds(row1, beg1, end1);
  int c0;
  float s0;
  edge_record<MODE>(p, beg0 + lane, end0, c0, s0);
  while (row0 < p.num_rows) {
    const int row2 = draw();
    int beg2, end2;
    bounds(row2, beg2, end2);
    int c1;
    float s1;
    edge_record<MODE>(p, beg1 + lane, end1, c1, s1);
    if (end0 >= 0) {
      const float r = p.rs ? __ldg(p.rs + row0) : 1.f;
      float acc[NACC][VEC];
#pragma unroll
      for (int k = 0; k < NACC; ++k) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[k][i] = 0.f;
      }
      sum_edges<T, VEC, NACC, MODE>(p, beg0, end0, 0, 1, lane, acc, c0, s0);
      store_row<T, VEC, NACC>(p, row0, lane, r, acc);
    }
    row0 = row1; beg0 = beg1; end0 = end1; c0 = c1; s0 = s1;
    row1 = row2; beg1 = beg2; end1 = end2;
  }
  if constexpr (GQ) {            // the last block to get here has seen every chunk drawn: rearm the queue
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(p.queue + 1, 1) == static_cast<int>(gridDim.x) - 1) {
      p.queue[0] = 0;
      p.queue[1] = 0;
      __threadfence();
    }
  }
  grid_dependency_wait();        // launched behind the hub kernel: complete only once the hub rows are written
}

template <typename T, int VEC, int NACC, int MODE>
__global__ void __launch_bounds__(kH16Threads) h16_rows_kernel(const H16Params<T> p) {
  rows_body<T, VEC, NACC, MODE, false>(p);
}

template <typename T, int VEC, int NACC, int MODE>
__global__ void __launch_bounds__(kH16Threads, 4) h16_queue_kernel(const H16Params<T> p) {
  rows_body<T, VEC, NACC, MODE, true>(p);
}

// Hub rows: one CTA per row of the hub list; warp w sums edge batches w, w + 16, ...; the 16 warp sums are added in
// warp order through shared memory, one chunk of the lane tile at a time.
template <typename T, int VEC, int NACC, int MODE>
__global__ void __launch_bounds__(kH16HubThreads) h16_hub_kernel(const H16Params<T> p) {
  // The row kernel runs behind this one as a programmatic dependent: let it start now, the two write disjoint rows.
  asm volatile("griddepcontrol.launch_dependents;");
  constexpr int WARPS = kH16HubThreads / 32;
  __shared__ float part[WARPS][32 * VEC];
  const int lane = threadIdx.x & 31;
  const int wid = threadIdx.x >> 5;
  const int n_hub = min(__ldg(p.hub_count), p.hub_capacity);
  for (int i = blockIdx.x; i < n_hub; i += gridDim.x) {
    const int row = __ldg(p.hub_rows + i);
    const int beg = __ldg(p.row_off + row);
    const int end = __ldg(p.row_off + row + 1);
    float acc[NACC][VEC];
#pragma unroll
    for (int k = 0; k < NACC; ++k) {
#pragma unroll
      for (int v = 0; v < VEC; ++v) acc[k][v] = 0.f;
    }
    int c;
    float s;
    edge_record<MODE>(p, beg + 32 * wid + lane, end, c, s);
    sum_edges<T, VEC, NACC, MODE>(p, beg, end, wid, WARPS, lane, acc, c, s);
    const float r = p.rs ? __ldg(p.rs + row) : 1.f;
#pragma unroll
    for (int k = 0; k < NACC; ++k) {
#pragma unroll
      for (int v = 0; v < VEC; ++v) part[wid][lane * VEC + v] = acc[k][v];
      __syncthreads();
      if (wid == 0) {
        float sum[1][VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          float t = part[0][lane * VEC + v];
          for (int w = 1; w < WARPS; ++w) t += part[w][lane * VEC + v];
          sum[0][v] = t;
        }
        const int o = (lane + 32 * k) * VEC;
        if (o < p.width) {
          float f[VEC];
#pragma unroll
          for (int v = 0; v < VEC; ++v) f[v] = sum[0][v] * r;
          __stcs(reinterpret_cast<typename Raw<VEC>::type*>(p.out + static_cast<size_t>(row) * p.ld + o), pack<T, VEC>(f));
        }
      }
      __syncthreads();             // part[] is rewritten by the next chunk / row
    }
  }
}

template <typename T, int VEC, int NACC, int MODE>
int launch_h16(const H16Params<T>& p, int num_edges, cudaStream_t stream) {
  const bool hubs = p.hub_threshold > 0 && p.hub_rows != nullptr;
  // as agg.cu: on a graph of 2^18 edges and more the row kernel starts while the hub rows are being summed
  const bool overlap = hubs && num_edges >= (1 << 18);
  if (hubs && p.hub_capacity > 0) {
    const int grid = std::min(p.hub_capacity, sm_count() * (num_edges >= (1 << 24) ? 1 : 2));
    h16_hub_kernel<T, VEC, NACC, MODE><<<grid, kH16HubThreads, 0, stream>>>(p);
    STG_LAUNCH_CHECK("h16_hub_kernel");
  }
  constexpr int warps = kH16Threads / 32;
  const int blocks = (p.num_rows + warps - 1) / warps;
  // the global row queue from two waves of warps on (agg.cu's threshold); a small graph keeps one row per warp
  if (p.queue != nullptr && p.num_rows >= 2 * sm_count() * 4 * warps) {
    const int grid = std::min(sm_count() * 4, blocks);
    STG_CUDA(launch_overlapped(h16_queue_kernel<T, VEC, NACC, MODE>, grid, kH16Threads, stream, overlap, p));
    STG_LAUNCH_CHECK("h16_queue_kernel");
  } else {
    STG_CUDA(launch_overlapped(h16_rows_kernel<T, VEC, NACC, MODE>, blocks, kH16Threads, stream, overlap, p));
    STG_LAUNCH_CHECK("h16_rows_kernel");
  }
  return STG_OK;
}

template <typename T, int VEC, int MODE>
int dispatch_h16(const H16Params<T>& p, int num_edges, cudaStream_t stream) {
  const int nvec = (p.width + VEC - 1) / VEC;
  if (nvec <= 32) return launch_h16<T, VEC, 1, MODE>(p, num_edges, stream);
  if (nvec <= 64) return launch_h16<T, VEC, 2, MODE>(p, num_edges, stream);
  return launch_h16<T, VEC, 4, MODE>(p, num_edges, stream);
}

template <typename T>
int agg_h16_device(const StgCsrView* g, const StgEdgeMeta* meta, const T* x, int feat, const float* ns, const float* es,
                   const float* rs, T* out, cudaStream_t stream) {
  H16Params<T> p;
  p.row_off = g->row_offset;
  p.col = g->column_indices;
  p.eids = g->eids;
  p.hub_rows = g->hub_rows;
  p.hub_count = g->hub_count;
  p.meta = reinterpret_cast<const int2*>(meta);
  p.queue = g->work_queue;
  p.num_rows = g->num_nodes;
  p.eid_base = g->eid_base;
  p.eids_identity = g->eids_identity;
  p.hub_threshold = (g->hub_rows && g->hub_count) ? g->hub_threshold : 0;
  p.hub_capacity = g->hub_capacity;
  p.ld = feat;
  p.ns = ns;
  p.es = es;
  p.rs = rs;
  const uintptr_t addr = reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out);
  int vec = 1;
  if (feat % 8 == 0 && (addr & 15u) == 0) vec = 8;
  else if (feat % 4 == 0 && (addr & 7u) == 0) vec = 4;
  else if (feat % 2 == 0 && (addr & 3u) == 0) vec = 2;
  const int chunk = 32 * 4 * vec;   // widest tile one launch covers
  for (int f0 = 0; f0 < feat; f0 += chunk) {
    p.x = x + f0;
    p.out = out + f0;
    p.width = std::min(chunk, feat - f0);
    int rc;
    if (meta != nullptr) {
      if (vec == 8) rc = dispatch_h16<T, 8, kH16Packed>(p, g->num_edges, stream);
      else if (vec == 4) rc = dispatch_h16<T, 4, kH16Packed>(p, g->num_edges, stream);
      else if (vec == 2) rc = dispatch_h16<T, 2, kH16Packed>(p, g->num_edges, stream);
      else rc = dispatch_h16<T, 1, kH16Packed>(p, g->num_edges, stream);
    } else {
      if (vec == 8) rc = dispatch_h16<T, 8, kH16Plain>(p, g->num_edges, stream);
      else if (vec == 4) rc = dispatch_h16<T, 4, kH16Plain>(p, g->num_edges, stream);
      else if (vec == 2) rc = dispatch_h16<T, 2, kH16Plain>(p, g->num_edges, stream);
      else rc = dispatch_h16<T, 1, kH16Plain>(p, g->num_edges, stream);
    }
    if (rc != STG_OK) return rc;
  }
  return STG_OK;
}

int agg_h16(const StgCsrView* g, const StgEdgeMeta* meta, const void* x, int32_t feat, int32_t dtype, const float* ns,
            const float* es, const float* rs, void* out, cudaStream_t stream) {
  if (dtype == STG_DTYPE_BF16)
    return agg_h16_device(g, meta, static_cast<const __nv_bfloat16*>(x), feat, ns, es, rs, static_cast<__nv_bfloat16*>(out),
                          stream);
  return agg_h16_device(g, meta, static_cast<const __half*>(x), feat, ns, es, rs, static_cast<__half*>(out), stream);
}

int check_h16_args(const StgCsrView* g, bool need_eids, int32_t feat, int32_t dtype) {
  const int rc = validate_view(g, need_eids);
  if (rc != STG_OK) return rc;
  STG_CHECK_ARG(feat >= 0, "feat must not be negative (got %d)", feat);
  STG_CHECK_ARG(dtype == STG_DTYPE_BF16 || dtype == STG_DTYPE_F16, "unknown dtype code %d (STG_DTYPE_BF16 = 1, STG_DTYPE_F16 = 2)",
                dtype);
  return STG_OK;
}

}  // namespace
}  // namespace stg

using namespace stg;

STG_API int stg_agg_scaled_sum_h16(const StgCsrView* g, const void* x, int32_t feat, int32_t dtype,
                                   const float* nbr_scale, const float* edge_scale, const float* row_scale, void* out,
                                   void* stream) {
  const int rc = check_h16_args(g, edge_scale != nullptr, feat, dtype);
  if (rc != STG_OK) return rc;
  if (g->num_nodes == 0 || feat == 0) return STG_OK;
  STG_CHECK_ARG(x != nullptr && out != nullptr, "x / out is NULL");
  STG_CHECK_ARG(x != out, "x and out must not alias");
  return agg_h16(g, nullptr, x, feat, dtype, nbr_scale, edge_scale, row_scale, out, as_stream(stream));
}

STG_API int stg_agg_packed_sum_h16(const StgCsrView* g, const StgEdgeMeta* meta, const void* x, int32_t feat,
                                   int32_t dtype, const float* row_scale, void* out, void* stream) {
  const int rc = check_h16_args(g, false, feat, dtype);
  if (rc != STG_OK) return rc;
  if (g->num_nodes == 0 || feat == 0) return STG_OK;
  STG_CHECK_ARG(g->num_edges == 0 || (meta != nullptr && aligned8(meta)),
                "meta must be a non-NULL, 8-byte aligned device pointer");
  STG_CHECK_ARG(x != nullptr && out != nullptr, "x / out is NULL");
  STG_CHECK_ARG(x != out, "x and out must not alias");
  // an empty graph has nothing to read through meta: the plain path writes the zero rows
  return agg_h16(g, g->num_edges == 0 ? nullptr : meta, x, feat, dtype, nullptr, nullptr, row_scale, out,
                 as_stream(stream));
}
