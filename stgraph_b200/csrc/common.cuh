// Shared helpers for the stgraph_b200 CUDA library (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/stgraph_b200.h"

#define STG_API extern "C" __attribute__((visibility("default")))

namespace stg {

// thread-local last-error text, read through stg_last_error()
void set_error(const char* fmt, ...);

#define STG_CHECK_ARG(cond, ...)                 \
  do {                                           \
    if (!(cond)) {                               \
      ::stg::set_error(__VA_ARGS__);             \
      return STG_ERR_INVALID_ARGUMENT;           \
    }                                            \
  } while (0)

#define STG_CUDA(call)                                                             \
  do {                                                                             \
    cudaError_t e_ = (call);                                                       \
    if (e_ != cudaSuccess) {                                                       \
      ::stg::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),    \
                       __FILE__, __LINE__);                                        \
      return STG_ERR_CUDA;                                                         \
    }                                                                              \
  } while (0)

#define STG_LAUNCH_CHECK(name)                                                     \
  do {                                                                             \
    cudaError_t e_ = cudaGetLastError();                                           \
    if (e_ != cudaSuccess) {                                                       \
      ::stg::set_error("launch of %s failed: %s", name, cudaGetErrorString(e_));   \
      return STG_ERR_CUDA;                                                         \
    }                                                                              \
  } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline bool aligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Checks every aggregation entry point makes on a CSR view before it launches anything.
inline int validate_view(const StgCsrView* g, bool need_eids) {
  STG_CHECK_ARG(g != nullptr, "graph view is NULL");
  STG_CHECK_ARG(g->num_nodes >= 0 && g->num_edges >= 0, "negative graph size (%d nodes, %d edges)",
                g->num_nodes, g->num_edges);
  STG_CHECK_ARG(g->row_offset != nullptr, "row_offset is NULL");
  STG_CHECK_ARG(g->num_edges == 0 || g->column_indices != nullptr, "column_indices is NULL");
  STG_CHECK_ARG(!need_eids || g->eids_identity || g->num_edges == 0 || g->eids != nullptr,
                "eids is NULL but an edge tensor is indexed by edge id");
  return STG_OK;
}

// Number of SMs of the current device (cached per process; 148 on B200).
int sm_count();

// ---- device helpers ------------------------------------------------------
__device__ __forceinline__ int ld_idx(const int32_t* p) { return __ldg(p); }

// streaming (evict-first) loads for data touched exactly once
__device__ __forceinline__ int ld_stream(const int32_t* p) { return __ldcs(p); }
__device__ __forceinline__ float ld_stream(const float* p) { return __ldcs(p); }

template <int VEC> struct VecT;
template <> struct VecT<1> { using type = float; };
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<4> { using type = float4; };

__device__ __forceinline__ void fma_vec(float& a, float s, float v) { a = fmaf(s, v, a); }
__device__ __forceinline__ void fma_vec(float2& a, float s, float2 v) {
  a.x = fmaf(s, v.x, a.x); a.y = fmaf(s, v.y, a.y);
}
__device__ __forceinline__ void fma_vec(float4& a, float s, float4 v) {
  a.x = fmaf(s, v.x, a.x); a.y = fmaf(s, v.y, a.y);
  a.z = fmaf(s, v.z, a.z); a.w = fmaf(s, v.w, a.w);
}
__device__ __forceinline__ void zero_vec(float& a) { a = 0.f; }
__device__ __forceinline__ void zero_vec(float2& a) { a = make_float2(0.f, 0.f); }
__device__ __forceinline__ void zero_vec(float4& a) { a = make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ void scale_vec(float& a, float s) { a *= s; }
__device__ __forceinline__ void scale_vec(float2& a, float s) { a.x *= s; a.y *= s; }
__device__ __forceinline__ void scale_vec(float4& a, float s) { a.x *= s; a.y *= s; a.z *= s; a.w *= s; }
__device__ __forceinline__ void add_vec(float& a, float b) { a += b; }
__device__ __forceinline__ void add_vec(float2& a, float2 b) { a.x += b.x; a.y += b.y; }
__device__ __forceinline__ void add_vec(float4& a, float4 b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }

// ---- programmatic dependent launch (hub kernel || row kernel) -----------------
// The row kernels run as programmatic dependents of the hub kernel (both in flight at once); a row
// kernel block does not retire before the hub kernel has completed and flushed, so "row kernel
// complete" implies "hub rows written" for whatever follows in the stream.
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Launch `kernel` so that it may start while the previous kernel of the stream is still running
// (programmatic dependent launch); the kernel orders itself with grid_dependency_wait().
template <typename... KArgs, typename... Args>
cudaError_t launch_overlapped(void (*kernel)(KArgs...), int blocks, int threads, cudaStream_t stream, bool overlap,
                              Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(blocks);
  cfg.blockDim = dim3(threads);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = overlap ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

}  // namespace stg
