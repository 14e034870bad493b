// Fused element-wise pieces of the TGCN (GRU) cell for sm_100a.
//
// Reference: stgraph/nn/pytorch/temporal/tgcn.py:21-47 computes, per time step, on [N, H] tensors
//     Z = sigmoid(linear_z([conv_z | H]))        R = sigmoid(linear_r([conv_r | H]))
//     H~ = tanh(linear_h([conv_h | H * R]))      H' = Z * H + (1 - Z) * H~
// with conv_* = clamp(GCNConv(X) , -1e6, 1e6) -- about sixteen separate element-wise kernels forward and thirty
// backward, each a full pass over [N, H] (config 4: N = 10^6, H = 64).  The GEMMs stay cuBLAS; what is left is three
// element-wise passes forward and three backward:
//     bias_clamp:  a = clamp(a + bias, lo, hi)                    (in place on the aggregation output [N, 3H])
//     reset:       hr = h * sigmoid(pr)
//     update:      out = z * h + (1 - z) * tanh(ph),  z = sigmoid(pz)
// Backward kernels recompute the activations from the saved pre-activations (no extra tensors are kept).
// HBM-roofline kernels: algorithmic bytes = 4 * (tensors read + tensors written) * N * H.
#include "common.cuh"
#include "h16.cuh"

#include <initializer_list>

namespace stg {
namespace {

constexpr int kGateThreads = 256;

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + __expf(-x)); }

inline int gate_blocks(int64_t n) {
  const int64_t b = (n + kGateThreads - 1) / kGateThreads;
  const int64_t cap = static_cast<int64_t>(sm_count()) * 16;
  return static_cast<int>(b < cap ? (b > 0 ? b : 1) : cap);
}

__global__ void __launch_bounds__(kGateThreads) bias_clamp_kernel(float* __restrict__ a, const float* __restrict__ bias,
                                                                 int64_t n, int cols, float lo, float hi) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    float v = a[i];
    if (bias) v += __ldg(bias + static_cast<int>(i % cols));
    a[i] = (v != v) ? v : fminf(fmaxf(v, lo), hi);      // NaN propagates, like torch.clamp (fminf / fmaxf drop it)
  }
}

// four elements per thread (cols % 4 == 0, 16-byte aligned): the bias index does not wrap inside a float4
__global__ void __launch_bounds__(kGateThreads) bias_clamp4_kernel(float4* __restrict__ a, const float* __restrict__ bias,
                                                                  int64_t n4, int cols, float lo, float hi) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v = a[i];
    if (bias) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(bias + static_cast<int>((i * 4) % cols)));
      v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
    }
    v.x = (v.x != v.x) ? v.x : fminf(fmaxf(v.x, lo), hi);
    v.y = (v.y != v.y) ? v.y : fminf(fmaxf(v.y, lo), hi);
    v.z = (v.z != v.z) ? v.z : fminf(fmaxf(v.z, lo), hi);
    v.w = (v.w != v.w) ? v.w : fminf(fmaxf(v.w, lo), hi);
    a[i] = v;
  }
}

// d_a = d_y where the clamped value lies strictly inside (lo, hi), else 0 (torch.clamp passes the gradient on the
// closed interval of the UNCLAMPED value; the two differ only when the pre-clamp value equals a bound exactly)
__global__ void __launch_bounds__(kGateThreads) clamp_bwd_kernel(const float* __restrict__ y, const float* __restrict__ d_y,
                                                                float* __restrict__ d_a, int64_t n, float lo, float hi) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float v = y[i];
    d_a[i] = (v > lo && v < hi) ? d_y[i] : 0.f;      // a NaN value gets no gradient, like torch.clamp's mask
  }
}

__global__ void __launch_bounds__(kGateThreads) reset_fwd_kernel(const float* __restrict__ pr, const float* __restrict__ h,
                                                                float* __restrict__ hr, int64_t n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
    hr[i] = h[i] * sigmoidf_(pr[i]);
}

__global__ void __launch_bounds__(kGateThreads) reset_bwd_kernel(const float* __restrict__ pr, const float* __restrict__ h,
                                                                const float* __restrict__ d_hr, float* __restrict__ d_pr,
                                                                float* __restrict__ d_h, int64_t n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float r = sigmoidf_(pr[i]);
    const float g = d_hr[i];
    d_pr[i] = g * h[i] * r * (1.f - r);
    d_h[i] = g * r;
  }
}

__global__ void __launch_bounds__(kGateThreads) update_fwd_kernel(const float* __restrict__ pz, const float* __restrict__ ph,
                                                                 const float* __restrict__ h, float* __restrict__ out,
                                                                 int64_t n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float z = sigmoidf_(pz[i]);
    out[i] = z * h[i] + (1.f - z) * tanhf(ph[i]);
  }
}

__global__ void __launch_bounds__(kGateThreads) update_bwd_kernel(const float* __restrict__ pz, const float* __restrict__ ph,
                                                                 const float* __restrict__ h, const float* __restrict__ d_out,
                                                                 float* __restrict__ d_pz, float* __restrict__ d_ph,
                                                                 float* __restrict__ d_h, int64_t n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float z = sigmoidf_(pz[i]);
    const float t = tanhf(ph[i]);
    const float g = d_out[i];
    d_pz[i] = g * (h[i] - t) * z * (1.f - z);
    d_ph[i] = g * (1.f - z) * (1.f - t * t);
    d_h[i] = g * z;
  }
}

// ---- the same gate arithmetic on the block layout of the one-Function cell (ops_tgcn.py): the three gate
// pre-activations are the column blocks (z | r | h) of ONE [rows, 3*hid] matrix p, so that every GEMM that produces or
// consumes them works on a column block in place and the bias / weight gradients are one reduction / one GEMM each.
// V = 4: one float4 per thread and step (hid % 4 == 0, 16-byte aligned bases); V = 1: scalar.
template <int V> struct GateVec;
template <> struct GateVec<1> {
  using T = float;
  static __device__ __forceinline__ void get(const T& v, float (&a)[1]) { a[0] = v; }
  static __device__ __forceinline__ T make(const float (&a)[1]) { return a[0]; }
};
template <> struct GateVec<4> {
  using T = float4;
  static __device__ __forceinline__ void get(const T& v, float (&a)[4]) { a[0] = v.x; a[1] = v.y; a[2] = v.z; a[3] = v.w; }
  static __device__ __forceinline__ T make(const float (&a)[4]) { return make_float4(a[0], a[1], a[2], a[3]); }
};
template <int V> __device__ __forceinline__ void ldg_v(const float* p, float (&a)[V]) {
  GateVec<V>::get(*reinterpret_cast<const typename GateVec<V>::T*>(p), a);
}
template <int V> __device__ __forceinline__ void st_v(float* p, const float (&a)[V]) {
  *reinterpret_cast<typename GateVec<V>::T*>(p) = GateVec<V>::make(a);
}

// i runs over the [rows, hid] elements in steps of V; q is the matching element of the z block of p / d_p
#define STG_CELL_LOOP(V)                                                                                           \
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x * V;                                          \
  for (int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * V; i < n; i += stride)

template <int V>
__global__ void __launch_bounds__(kGateThreads) cell_reset_fwd_kernel(const float* __restrict__ p, const float* __restrict__ h,
                                                                     float* __restrict__ hr, int64_t n, int hid) {
  STG_CELL_LOOP(V) {
    const int64_t r = i / hid;
    const int64_t q = r * 3 * hid + (i - r * hid);
    float pr[V], hv[V], o[V];
    ldg_v<V>(p + q + hid, pr);
    ldg_v<V>(h + i, hv);
#pragma unroll
    for (int k = 0; k < V; ++k) o[k] = hv[k] * sigmoidf_(pr[k]);
    st_v<V>(hr + i, o);
  }
}

// d_p[:, r block] = d_hr * h * r * (1 - r);  d_h += d_hr * r   (d_h already holds the update gate's share)
template <int V>
__global__ void __launch_bounds__(kGateThreads) cell_reset_bwd_kernel(const float* __restrict__ p, const float* __restrict__ h,
                                                                     const float* __restrict__ d_hr, float* __restrict__ d_p,
                                                                     float* __restrict__ d_h, int64_t n, int hid) {
  STG_CELL_LOOP(V) {
    const int64_t r = i / hid;
    const int64_t q = r * 3 * hid + (i - r * hid) + hid;
    float pr[V], hv[V], g[V], dh[V], dp[V];
    ldg_v<V>(p + q, pr);
    ldg_v<V>(h + i, hv);
    ldg_v<V>(d_hr + i, g);
    ldg_v<V>(d_h + i, dh);
#pragma unroll
    for (int k = 0; k < V; ++k) {
      const float s = sigmoidf_(pr[k]);
      dp[k] = g[k] * hv[k] * s * (1.f - s);
      dh[k] += g[k] * s;
    }
    st_v<V>(d_p + q, dp);
    st_v<V>(d_h + i, dh);
  }
}

template <int V>
__global__ void __launch_bounds__(kGateThreads) cell_update_fwd_kernel(const float* __restrict__ p, const float* __restrict__ h,
                                                                      float* __restrict__ out, int64_t n, int hid) {
  STG_CELL_LOOP(V) {
    const int64_t r = i / hid;
    const int64_t q = r * 3 * hid + (i - r * hid);
    float pz[V], ph[V], hv[V], o[V];
    ldg_v<V>(p + q, pz);
    ldg_v<V>(p + q + 2 * hid, ph);
    ldg_v<V>(h + i, hv);
#pragma unroll
    for (int k = 0; k < V; ++k) {
      const float z = sigmoidf_(pz[k]);
      o[k] = z * hv[k] + (1.f - z) * tanhf(ph[k]);
    }
    st_v<V>(out + i, o);
  }
}

// d_p[:, z block], d_p[:, h block] and d_h = d_out * z (the reset gate's share is added by cell_reset_bwd_kernel)
template <int V>
__global__ void __launch_bounds__(kGateThreads) cell_update_bwd_kernel(const float* __restrict__ p, const float* __restrict__ h,
                                                                      const float* __restrict__ d_out, float* __restrict__ d_p,
                                                                      float* __restrict__ d_h, int64_t n, int hid) {
  STG_CELL_LOOP(V) {
    const int64_t r = i / hid;
    const int64_t q = r * 3 * hid + (i - r * hid);
    float pz[V], ph[V], hv[V], g[V], dz[V], dc[V], dh[V];
    ldg_v<V>(p + q, pz);
    ldg_v<V>(p + q + 2 * hid, ph);
    ldg_v<V>(h + i, hv);
    ldg_v<V>(d_out + i, g);
#pragma unroll
    for (int k = 0; k < V; ++k) {
      const float z = sigmoidf_(pz[k]);
      const float t = tanhf(ph[k]);
      dz[k] = g[k] * (hv[k] - t) * z * (1.f - z);
      dc[k] = g[k] * (1.f - z) * (1.f - t * t);
      dh[k] = g[k] * z;
    }
    st_v<V>(d_p + q, dz);
    st_v<V>(d_p + q + 2 * hid, dc);
    st_v<V>(d_h + i, dh);
  }
}

// ---- the 16-bit cell (ops_tgcn.py under torch.autocast): the tensors that are GEMM operands are stored as FT
// (__nv_bfloat16 / __half), everything else stays fp32.  The arithmetic is the fp32 kernels', in the same order, on the
// widened values; a value is rounded once, when it is stored to an FT tensor.  V = 4: 8-byte FT and 16-byte fp32 accesses.
template <typename FT, int V> __device__ __forceinline__ void ldg_h(const FT* p, float (&a)[V]) {
  unpack<FT, V>(*reinterpret_cast<const typename Raw<V>::type*>(p), a);
}
template <typename FT, int V> __device__ __forceinline__ void st_h(FT* p, const float (&a)[V]) {
  *reinterpret_cast<typename Raw<V>::type*>(p) = pack<FT, V>(a);
}

// y = clamp(a + bias[col], lo, hi) rounded once; a is the 16-bit aggregation output and is kept (the backward recomputes
// the clamp mask from it).  y may be a.
template <typename FT, int V>
__global__ void __launch_bounds__(kGateThreads) cell_bias_clamp16_kernel(const FT* a, const float* __restrict__ bias, FT* y,
                                                                         int64_t n, int cols, float lo, float hi) {
  STG_CELL_LOOP(V) {
    float v[V];
    ldg_h<FT, V>(a + i, v);
    if (bias) {
      float b[V];
      ldg_v<V>(bias + static_cast<int>(i % cols), b);
#pragma unroll
      for (int k = 0; k < V; ++k) v[k] += b[k];
    }
#pragma unroll
    for (int k = 0; k < V; ++k) v[k] = (v[k] != v[k]) ? v[k] : fminf(fmaxf(v[k], lo), hi);
    st_h<FT, V>(y + i, v);
  }
}

// d_a = d_y where lo < a + bias[col] < hi in fp32 (the fp32 cell's mask on its unrounded clamp input), else 0.  The mask
// is NOT taken from the rounded y: bf16 rounds 1e6 to 999424 < 1e6.  d_y's bits are passed through; d_a may be d_y.
template <typename FT, int V>
__global__ void __launch_bounds__(kGateThreads) cell_clamp_bwd16_kernel(const FT* __restrict__ a, const float* __restrict__ bias,
                                                                        const FT* d_y, FT* d_a, int64_t n, int cols, float lo,
                                                                        float hi) {
  STG_CELL_LOOP(V) {
    float v[V];
    ldg_h<FT, V>(a + i, v);
    if (bias) {
      float b[V];
      ldg_v<V>(bias + static_cast<int>(i % cols), b);
#pragma unroll
      for (int k = 0; k < V; ++k) v[k] += b[k];
    }
    typename Raw<V>::type g = *reinterpret_cast<const typename Raw<V>::type*>(d_y + i);
    unsigned short* w = reinterpret_cast<unsigned short*>(&g);
#pragma unroll
    for (int k = 0; k < V; ++k) w[k] = (v[k] > lo && v[k] < hi) ? w[k] : static_cast<unsigned short>(0);
    *reinterpret_cast<typename Raw<V>::type*>(d_a + i) = g;
  }
}

// hr = h * sigmoid(p_r), stored as FT (hr is only the operand of the candidate-state GEMM)
template <typename FT, int V>
__global__ void __launch_bounds__(kGateThreads) cell_reset_fwd16_kernel(const float* __restrict__ p, const float* __restrict__ h,
                                                                        FT* __restrict__ hr, int64_t n, int hid) {
  STG_CELL_LOOP(V) {
    const int64_t r = i / hid;
    const int64_t q = r * 3 * hid + (i - r * hid);
    float pr[V], hv[V], o[V];
    ldg_v<V>(p + q + hid, pr);
    ldg_v<V>(h + i, hv);
#pragma unroll
    for (int k = 0; k < V; ++k) o[k] = hv[k] * sigmoidf_(pr[k]);
    st_h<FT, V>(hr + i, o);
  }
}

// cell_reset_bwd_kernel, and the r block of d_p once more as FT in d_p16 (the operand of the backward GEMMs)
template <typename FT, int V>
__global__ void __launch_bounds__(kGateThreads) cell_reset_bwd16_kernel(const float* __restrict__ p, const float* __restrict__ h,
                                                                        const float* __restrict__ d_hr, float* __restrict__ d_p,
                                                                        FT* __restrict__ d_p16, float* __restrict__ d_h,
                                                                        int64_t n, int hid) {
  STG_CELL_LOOP(V) {
    const int64_t r = i / hid;
    const int64_t q = r * 3 * hid + (i - r * hid) + hid;
    float pr[V], hv[V], g[V], dh[V], dp[V];
    ldg_v<V>(p + q, pr);
    ldg_v<V>(h + i, hv);
    ldg_v<V>(d_hr + i, g);
    ldg_v<V>(d_h + i, dh);
#pragma unroll
    for (int k = 0; k < V; ++k) {
      const float s = sigmoidf_(pr[k]);
      dp[k] = g[k] * hv[k] * s * (1.f - s);
      dh[k] += g[k] * s;
    }
    st_v<V>(d_p + q, dp);
    st_h<FT, V>(d_p16 + q, dp);
    st_v<V>(d_h + i, dh);
  }
}

// cell_update_bwd_kernel, and the z and h blocks of d_p once more as FT in d_p16
template <typename FT, int V>
__global__ void __launch_bounds__(kGateThreads) cell_update_bwd16_kernel(const float* __restrict__ p, const float* __restrict__ h,
                                                                         const float* __restrict__ d_out, float* __restrict__ d_p,
                                                                         FT* __restrict__ d_p16, float* __restrict__ d_h,
                                                                         int64_t n, int hid) {
  STG_CELL_LOOP(V) {
    const int64_t r = i / hid;
    const int64_t q = r * 3 * hid + (i - r * hid);
    float pz[V], ph[V], hv[V], g[V], dz[V], dc[V], dh[V];
    ldg_v<V>(p + q, pz);
    ldg_v<V>(p + q + 2 * hid, ph);
    ldg_v<V>(h + i, hv);
    ldg_v<V>(d_out + i, g);
#pragma unroll
    for (int k = 0; k < V; ++k) {
      const float z = sigmoidf_(pz[k]);
      const float t = tanhf(ph[k]);
      dz[k] = g[k] * (hv[k] - t) * z * (1.f - z);
      dc[k] = g[k] * (1.f - z) * (1.f - t * t);
      dh[k] = g[k] * z;
    }
    st_v<V>(d_p + q, dz);
    st_v<V>(d_p + q + 2 * hid, dc);
    st_h<FT, V>(d_p16 + q, dz);
    st_h<FT, V>(d_p16 + q + 2 * hid, dc);
    st_v<V>(d_h + i, dh);
  }
}
#undef STG_CELL_LOOP

template <class... P>
inline bool cell_vec_ok(int hid, P... ptrs) {
  return hid % 4 == 0 && (aligned16(ptrs) && ...);
}

// f(FT*{}) with FT the storage type of StgDtype code dtype (checked by the caller)
template <class F> inline void with_h16(int32_t dtype, F&& f) {
  if (dtype == STG_DTYPE_BF16) f(static_cast<__nv_bfloat16*>(nullptr));
  else f(static_cast<__half*>(nullptr));
}

// four lanes: width % 4 == 0, fp32 bases 16-byte and 16-bit bases 8-byte aligned
inline bool vec16_ok(int width, std::initializer_list<const void*> f32, std::initializer_list<const void*> h16) {
  if (width % 4 != 0) return false;
  for (const void* p : f32)
    if (!aligned16(p)) return false;
  for (const void* p : h16)
    if (!aligned8(p)) return false;
  return true;
}

}  // namespace
}  // namespace stg

using namespace stg;

STG_API int stg_tgcn_reset_fwd_f32(const float* p, const float* h, float* hr, int64_t rows, int32_t hid, void* stream) {
  STG_CHECK_ARG(rows >= 0 && hid > 0, "bad shape (%lld x %d)", static_cast<long long>(rows), hid);
  if (rows == 0) return STG_OK;
  STG_CHECK_ARG(p && h && hr, "NULL tensor");
  const int64_t n = rows * hid;
  if (cell_vec_ok(hid, p, h, hr)) cell_reset_fwd_kernel<4><<<gate_blocks(n / 4), kGateThreads, 0, as_stream(stream)>>>(p, h, hr, n, hid);
  else cell_reset_fwd_kernel<1><<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(p, h, hr, n, hid);
  STG_LAUNCH_CHECK("cell_reset_fwd_kernel");
  return STG_OK;
}

STG_API int stg_tgcn_reset_bwd_f32(const float* p, const float* h, const float* d_hr, float* d_p, float* d_h, int64_t rows,
                                   int32_t hid, void* stream) {
  STG_CHECK_ARG(rows >= 0 && hid > 0, "bad shape (%lld x %d)", static_cast<long long>(rows), hid);
  if (rows == 0) return STG_OK;
  STG_CHECK_ARG(p && h && d_hr && d_p && d_h, "NULL tensor");
  const int64_t n = rows * hid;
  if (cell_vec_ok(hid, p, h, d_hr, d_p, d_h))
    cell_reset_bwd_kernel<4><<<gate_blocks(n / 4), kGateThreads, 0, as_stream(stream)>>>(p, h, d_hr, d_p, d_h, n, hid);
  else cell_reset_bwd_kernel<1><<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(p, h, d_hr, d_p, d_h, n, hid);
  STG_LAUNCH_CHECK("cell_reset_bwd_kernel");
  return STG_OK;
}

STG_API int stg_tgcn_update_fwd_f32(const float* p, const float* h, float* out, int64_t rows, int32_t hid, void* stream) {
  STG_CHECK_ARG(rows >= 0 && hid > 0, "bad shape (%lld x %d)", static_cast<long long>(rows), hid);
  if (rows == 0) return STG_OK;
  STG_CHECK_ARG(p && h && out, "NULL tensor");
  const int64_t n = rows * hid;
  if (cell_vec_ok(hid, p, h, out)) cell_update_fwd_kernel<4><<<gate_blocks(n / 4), kGateThreads, 0, as_stream(stream)>>>(p, h, out, n, hid);
  else cell_update_fwd_kernel<1><<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(p, h, out, n, hid);
  STG_LAUNCH_CHECK("cell_update_fwd_kernel");
  return STG_OK;
}

STG_API int stg_tgcn_update_bwd_f32(const float* p, const float* h, const float* d_out, float* d_p, float* d_h, int64_t rows,
                                    int32_t hid, void* stream) {
  STG_CHECK_ARG(rows >= 0 && hid > 0, "bad shape (%lld x %d)", static_cast<long long>(rows), hid);
  if (rows == 0) return STG_OK;
  STG_CHECK_ARG(p && h && d_out && d_p && d_h, "NULL tensor");
  const int64_t n = rows * hid;
  if (cell_vec_ok(hid, p, h, d_out, d_p, d_h))
    cell_update_bwd_kernel<4><<<gate_blocks(n / 4), kGateThreads, 0, as_stream(stream)>>>(p, h, d_out, d_p, d_h, n, hid);
  else cell_update_bwd_kernel<1><<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(p, h, d_out, d_p, d_h, n, hid);
  STG_LAUNCH_CHECK("cell_update_bwd_kernel");
  return STG_OK;
}

STG_API int stg_bias_clamp_f32(float* a, const float* bias, int64_t rows, int32_t cols, float lo, float hi, void* stream) {
  STG_CHECK_ARG(rows >= 0 && cols > 0, "bad shape (%lld x %d)", static_cast<long long>(rows), cols);
  STG_CHECK_ARG(lo <= hi, "clamp bounds out of order");
  if (rows == 0) return STG_OK;
  STG_CHECK_ARG(a != nullptr, "a is NULL");
  const int64_t n = rows * cols;
  if (cols % 4 == 0 && aligned16(a) && (bias == nullptr || aligned16(bias)))
    bias_clamp4_kernel<<<gate_blocks(n / 4), kGateThreads, 0, as_stream(stream)>>>(reinterpret_cast<float4*>(a), bias, n / 4, cols,
                                                                                 lo, hi);
  else bias_clamp_kernel<<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(a, bias, n, cols, lo, hi);
  STG_LAUNCH_CHECK("bias_clamp_kernel");
  return STG_OK;
}

STG_API int stg_clamp_bwd_f32(const float* y, const float* d_y, float* d_a, int64_t n, float lo, float hi, void* stream) {
  STG_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return STG_OK;
  STG_CHECK_ARG(y && d_y && d_a, "NULL tensor");
  clamp_bwd_kernel<<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(y, d_y, d_a, n, lo, hi);
  STG_LAUNCH_CHECK("clamp_bwd_kernel");
  return STG_OK;
}

// ---- 16-bit cell: the same argument checks as the fp32 twins, plus the dtype code, all before any launch
#define STG_CHECK_DTYPE16(dtype)                                                                                  \
  STG_CHECK_ARG((dtype) == STG_DTYPE_BF16 || (dtype) == STG_DTYPE_F16,                                             \
                "unknown dtype code %d (STG_DTYPE_BF16 = 1, STG_DTYPE_F16 = 2)", (dtype))

STG_API int stg_tgcn_bias_clamp_h16(const void* a, const float* bias, void* y, int64_t rows, int32_t cols, int32_t dtype,
                                    float lo, float hi, void* stream) {
  STG_CHECK_ARG(rows >= 0 && cols > 0, "bad shape (%lld x %d)", static_cast<long long>(rows), cols);
  STG_CHECK_ARG(lo <= hi, "clamp bounds out of order");
  STG_CHECK_DTYPE16(dtype);
  if (rows == 0) return STG_OK;
  STG_CHECK_ARG(a != nullptr, "a is NULL");
  STG_CHECK_ARG(y != nullptr, "NULL tensor");
  const int64_t n = rows * cols;
  const bool vec = vec16_ok(cols, {bias}, {a, y});
  with_h16(dtype, [&](auto tag) {
    using FT = std::remove_pointer_t<decltype(tag)>;
    const FT* a_ = static_cast<const FT*>(a);
    FT* y_ = static_cast<FT*>(y);
    if (vec) cell_bias_clamp16_kernel<FT, 4><<<gate_blocks(n / 4), kGateThreads, 0, as_stream(stream)>>>(a_, bias, y_, n, cols, lo, hi);
    else cell_bias_clamp16_kernel<FT, 1><<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(a_, bias, y_, n, cols, lo, hi);
  });
  STG_LAUNCH_CHECK("cell_bias_clamp16_kernel");
  return STG_OK;
}

STG_API int stg_tgcn_clamp_bwd_h16(const void* a, const float* bias, const void* d_y, void* d_a, int64_t rows, int32_t cols,
                                   int32_t dtype, float lo, float hi, void* stream) {
  STG_CHECK_ARG(rows >= 0 && cols > 0, "bad shape (%lld x %d)", static_cast<long long>(rows), cols);
  STG_CHECK_ARG(lo <= hi, "clamp bounds out of order");
  STG_CHECK_DTYPE16(dtype);
  if (rows == 0) return STG_OK;
  STG_CHECK_ARG(a && d_y && d_a, "NULL tensor");
  const int64_t n = rows * cols;
  const bool vec = vec16_ok(cols, {bias}, {a, d_y, d_a});
  with_h16(dtype, [&](auto tag) {
    using FT = std::remove_pointer_t<decltype(tag)>;
    const FT* a_ = static_cast<const FT*>(a);
    const FT* g_ = static_cast<const FT*>(d_y);
    FT* d_ = static_cast<FT*>(d_a);
    if (vec) cell_clamp_bwd16_kernel<FT, 4><<<gate_blocks(n / 4), kGateThreads, 0, as_stream(stream)>>>(a_, bias, g_, d_, n, cols, lo, hi);
    else cell_clamp_bwd16_kernel<FT, 1><<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(a_, bias, g_, d_, n, cols, lo, hi);
  });
  STG_LAUNCH_CHECK("cell_clamp_bwd16_kernel");
  return STG_OK;
}

STG_API int stg_tgcn_reset_fwd_h16(const float* p, const float* h, void* hr, int64_t rows, int32_t hid, int32_t dtype,
                                   void* stream) {
  STG_CHECK_ARG(rows >= 0 && hid > 0, "bad shape (%lld x %d)", static_cast<long long>(rows), hid);
  STG_CHECK_DTYPE16(dtype);
  if (rows == 0) return STG_OK;
  STG_CHECK_ARG(p && h && hr, "NULL tensor");
  const int64_t n = rows * hid;
  const bool vec = vec16_ok(hid, {p, h}, {hr});
  with_h16(dtype, [&](auto tag) {
    using FT = std::remove_pointer_t<decltype(tag)>;
    FT* hr_ = static_cast<FT*>(hr);
    if (vec) cell_reset_fwd16_kernel<FT, 4><<<gate_blocks(n / 4), kGateThreads, 0, as_stream(stream)>>>(p, h, hr_, n, hid);
    else cell_reset_fwd16_kernel<FT, 1><<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(p, h, hr_, n, hid);
  });
  STG_LAUNCH_CHECK("cell_reset_fwd16_kernel");
  return STG_OK;
}

STG_API int stg_tgcn_reset_bwd_h16(const float* p, const float* h, const float* d_hr, float* d_p, void* d_p16, float* d_h,
                                   int64_t rows, int32_t hid, int32_t dtype, void* stream) {
  STG_CHECK_ARG(rows >= 0 && hid > 0, "bad shape (%lld x %d)", static_cast<long long>(rows), hid);
  STG_CHECK_DTYPE16(dtype);
  if (rows == 0) return STG_OK;
  STG_CHECK_ARG(p && h && d_hr && d_p && d_p16 && d_h, "NULL tensor");
  const int64_t n = rows * hid;
  const bool vec = vec16_ok(hid, {p, h, d_hr, d_p, d_h}, {d_p16});
  with_h16(dtype, [&](auto tag) {
    using FT = std::remove_pointer_t<decltype(tag)>;
    FT* q_ = static_cast<FT*>(d_p16);
    if (vec) cell_reset_bwd16_kernel<FT, 4><<<gate_blocks(n / 4), kGateThreads, 0, as_stream(stream)>>>(p, h, d_hr, d_p, q_, d_h, n, hid);
    else cell_reset_bwd16_kernel<FT, 1><<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(p, h, d_hr, d_p, q_, d_h, n, hid);
  });
  STG_LAUNCH_CHECK("cell_reset_bwd16_kernel");
  return STG_OK;
}

STG_API int stg_tgcn_update_bwd_h16(const float* p, const float* h, const float* d_out, float* d_p, void* d_p16, float* d_h,
                                    int64_t rows, int32_t hid, int32_t dtype, void* stream) {
  STG_CHECK_ARG(rows >= 0 && hid > 0, "bad shape (%lld x %d)", static_cast<long long>(rows), hid);
  STG_CHECK_DTYPE16(dtype);
  if (rows == 0) return STG_OK;
  STG_CHECK_ARG(p && h && d_out && d_p && d_p16 && d_h, "NULL tensor");
  const int64_t n = rows * hid;
  const bool vec = vec16_ok(hid, {p, h, d_out, d_p, d_h}, {d_p16});
  with_h16(dtype, [&](auto tag) {
    using FT = std::remove_pointer_t<decltype(tag)>;
    FT* q_ = static_cast<FT*>(d_p16);
    if (vec) cell_update_bwd16_kernel<FT, 4><<<gate_blocks(n / 4), kGateThreads, 0, as_stream(stream)>>>(p, h, d_out, d_p, q_, d_h, n, hid);
    else cell_update_bwd16_kernel<FT, 1><<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(p, h, d_out, d_p, q_, d_h, n, hid);
  });
  STG_LAUNCH_CHECK("cell_update_bwd16_kernel");
  return STG_OK;
}
#undef STG_CHECK_DTYPE16

STG_API int stg_gru_reset_fwd_f32(const float* pr, const float* h, float* hr, int64_t n, void* stream) {
  STG_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return STG_OK;
  STG_CHECK_ARG(pr && h && hr, "NULL tensor");
  reset_fwd_kernel<<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(pr, h, hr, n);
  STG_LAUNCH_CHECK("reset_fwd_kernel");
  return STG_OK;
}

STG_API int stg_gru_reset_bwd_f32(const float* pr, const float* h, const float* d_hr, float* d_pr, float* d_h, int64_t n,
                                  void* stream) {
  STG_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return STG_OK;
  STG_CHECK_ARG(pr && h && d_hr && d_pr && d_h, "NULL tensor");
  reset_bwd_kernel<<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(pr, h, d_hr, d_pr, d_h, n);
  STG_LAUNCH_CHECK("reset_bwd_kernel");
  return STG_OK;
}

STG_API int stg_gru_update_fwd_f32(const float* pz, const float* ph, const float* h, float* out, int64_t n, void* stream) {
  STG_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return STG_OK;
  STG_CHECK_ARG(pz && ph && h && out, "NULL tensor");
  update_fwd_kernel<<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(pz, ph, h, out, n);
  STG_LAUNCH_CHECK("update_fwd_kernel");
  return STG_OK;
}

STG_API int stg_gru_update_bwd_f32(const float* pz, const float* ph, const float* h, const float* d_out, float* d_pz,
                                   float* d_ph, float* d_h, int64_t n, void* stream) {
  STG_CHECK_ARG(n >= 0, "negative size");
  if (n == 0) return STG_OK;
  STG_CHECK_ARG(pz && ph && h && d_out && d_pz && d_ph && d_h, "NULL tensor");
  update_bwd_kernel<<<gate_blocks(n), kGateThreads, 0, as_stream(stream)>>>(pz, ph, h, d_out, d_pz, d_ph, d_h, n);
  STG_LAUNCH_CHECK("update_bwd_kernel");
  return STG_OK;
}
