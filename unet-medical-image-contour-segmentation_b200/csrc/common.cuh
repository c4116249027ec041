// Shared helpers for libunetb200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>
#include <type_traits>

#include "../../include/unetb200.h"

namespace ub {

typedef __nv_bfloat16 bf16;

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define UB_CHECK_ARG(cond, ...)                \
  do {                                         \
    if (!(cond)) {                             \
      ub::set_error(__VA_ARGS__);              \
      return UNETB200_E_INVALID;               \
    }                                          \
  } while (0)

#define UB_DTYPE_OK(dt) UB_CHECK_ARG((dt) == UNETB200_F32 || (dt) == UNETB200_BF16, "unsupported dtype %d", (int)(dt))

// ---- host-side dispatch: the runtime values an ABI call receives -> template arguments ------------------------
// Each helper calls `f` once with a tag that carries the choice in its type: a value of the chosen storage type
// (`using T = decltype(t);`) or a std::integral_constant (usable as a template argument as it is).  The last
// candidate of a list catches every value no earlier one matches, so a launcher validates its arguments first.

template <typename T>
struct dtype_code;
template <>
struct dtype_code<float> : std::integral_constant<int, UNETB200_F32> {};
template <>
struct dtype_code<bf16> : std::integral_constant<int, UNETB200_BF16> {};
template <>
struct dtype_code<long long> : std::integral_constant<int, UNETB200_I64> {};
template <>
struct dtype_code<uint8_t> : std::integral_constant<int, UNETB200_U8> {};

// the first of T, Rest... whose dtype code is `code`, else the last
template <typename T, typename... Rest, typename F>
inline void with_type(int code, F&& f) {
  if constexpr (sizeof...(Rest) == 0)
    f(T{});
  else if (code == dtype_code<T>::value)
    f(T{});
  else
    with_type<Rest...>(code, f);
}

// element (activation) storage type: bf16 for UNETB200_BF16, float otherwise
template <typename F>
inline void with_elem(int dtype, F&& f) {
  with_type<bf16, float>(dtype, f);
}

// the first of I, Rest... equal to `v`, else the last
template <int I, int... Rest, typename F>
inline void with_int(int v, F&& f) {
  if constexpr (sizeof...(Rest) == 0)
    f(std::integral_constant<int, I>{});
  else if (v == I)
    f(std::integral_constant<int, I>{});
  else
    with_int<Rest...>(v, f);
}

// vector width: V elements per access when `vec`, else 1
template <int V, typename F>
inline void with_vec(bool vec, F&& f) {
  with_int<V, 1>(vec ? V : 1, f);
}

template <typename F>
inline void with_bool(bool b, F&& f) {
  if (b)
    f(std::true_type{});
  else
    f(std::false_type{});
}

#define UB_LAUNCH_CHECK(what)                              \
  do {                                                     \
    cudaError_t e__ = cudaGetLastError();                  \
    if (e__ != cudaSuccess) return ub::cuda_fail(e__, what); \
  } while (0)

int sm_count();
// cudaFuncAttributeMaxDynamicSharedMemorySize for `func`, applied once per (device, function) under a mutex: forward
// runs on the Python main thread, backward on the autograd engine's device thread, and one process may drive
// several GPUs (the attribute is per device).
int set_max_dynamic_smem(const void* func, int bytes, const char* what);

template <typename T>
struct Elem;
template <>
struct Elem<float> {
  static __device__ __forceinline__ float ld(const float* p) { return *p; }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
  static __device__ __forceinline__ float round(float v) { return v; }
};
template <>
struct Elem<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
  static __device__ __forceinline__ float round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
};

// 8 consecutive elements <-> 8 floats, 16-byte (bf16) or 2x16-byte (fp32) accesses
__device__ __forceinline__ void load8(const float* p, float v[8]) {
  float4 a = *reinterpret_cast<const float4*>(p);
  float4 b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void load8(const __nv_bfloat16* p, float v[8]) {
  uint4 r = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ void store8(float* p, const float v[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void store8(__nv_bfloat16* p, const float v[8]) {
  uint4 r;
  r.x = pack_bf16x2(v[0], v[1]);
  r.y = pack_bf16x2(v[2], v[3]);
  r.z = pack_bf16x2(v[4], v[5]);
  r.w = pack_bf16x2(v[6], v[7]);
  *reinterpret_cast<uint4*>(p) = r;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace ub
