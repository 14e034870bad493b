// 16-bit feature rows (bf16 / fp16) for the kernels that read and write them with fp32 arithmetic (agg_h16.cu, gat.cu).
// An element is widened to fp32 when it is loaded and rounded to nearest even once, when it is stored.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

namespace stg {

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

}  // namespace stg
