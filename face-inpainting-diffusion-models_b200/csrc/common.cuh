// Shared helpers for the fidm_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/fidm_b200.h"

namespace fidm {

void set_error(const char* fmt, ...);

#define FIDM_REQUIRE(cond, code, ...)                   \
  do {                                                  \
    if (!(cond)) {                                      \
      ::fidm::set_error(__VA_ARGS__);                   \
      return (code);                                    \
    }                                                   \
  } while (0)

// Call after a kernel launch.  Returns a cudaError_t (>0) through the C ABI.
#define FIDM_CHECK_LAUNCH(what)                                                    \
  do {                                                                             \
    cudaError_t e__ = cudaGetLastError();                                          \
    if (e__ != cudaSuccess) {                                                      \
      ::fidm::set_error("%s: %s", (what), cudaGetErrorString(e__));                \
      return (int)e__;                                                             \
    }                                                                              \
  } while (0)

#define FIDM_CUDA(call)                                                            \
  do {                                                                             \
    cudaError_t e__ = (call);                                                      \
    if (e__ != cudaSuccess) {                                                      \
      ::fidm::set_error("%s: %s", #call, cudaGetErrorString(e__));                 \
      return (int)e__;                                                             \
    }                                                                              \
  } while (0)

constexpr int kMaxDevices = 64;
inline int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return (dev >= 0 && dev < kMaxDevices) ? dev : 0;
}
// SM count of the CURRENT device (cached per device ordinal: one process may drive several GPUs).
inline int num_sms() {
  static int n[kMaxDevices] = {};
  const int dev = current_device();
  if (n[dev] == 0) {
    int v = 0;
    cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
    n[dev] = v > 0 ? v : 148;
  }
  return n[dev];
}
// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute of a kernel: set it once per (kernel
// instantiation, device).  `flags` is a function-local static array of kMaxDevices bools owned by the caller.
template <typename F>
inline cudaError_t ensure_dynamic_smem(F kernel, int bytes, bool (&flags)[kMaxDevices]) {
  const int dev = current_device();
  if (flags[dev]) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) flags[dev] = true;
  return e;
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// fp16 stores saturate (cvt.satfinite): a normalized operand beyond 65504 clamps instead of becoming inf
template <> __device__ __forceinline__ __half from_f32<__half>(float v) {
  unsigned short r;
  asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(r) : "f"(v));
  return __ushort_as_half(r);
}

// A vector of V elements of T, loaded/stored with one instruction when it is 4/8/16 bytes.
template <typename T, int V> struct alignas(sizeof(T) * V) Vec { T v[V]; };

template <typename T, int V>
__device__ __forceinline__ void load_vec(const T* p, float (&out)[V]) {
  Vec<T, V> t = *reinterpret_cast<const Vec<T, V>*>(p);
#pragma unroll
  for (int i = 0; i < V; ++i) out[i] = to_f32<T>(t.v[i]);
}
template <typename T, int V>
__device__ __forceinline__ void store_vec(T* p, const float (&in)[V]) {
  Vec<T, V> t;
#pragma unroll
  for (int i = 0; i < V; ++i) t.v[i] = from_f32<T>(in[i]);
  *reinterpret_cast<Vec<T, V>*>(p) = t;
}

// ---- division by a launch-time constant without the ~25-instruction I2F / MUFU.RCP sequence (the single-thread TMA
// producers and MMA issuers of the tensor-core kernels are latency-bound on exactly that arithmetic):
//   n / d == (umulhi(mul, n) + n) >> sh   for 0 <= n < 2^31,  sh = ceil(log2 d),  mul = floor(2^32 (2^sh - d) / d) + 1
struct FastDiv { uint32_t d, mul, sh; };
inline FastDiv make_fastdiv(int d) {
  FastDiv f;
  f.d = (uint32_t)d;
  f.sh = 0;
  while ((1u << f.sh) < (uint32_t)d) ++f.sh;
  f.mul = (uint32_t)((((unsigned long long)1 << 32) * ((1ull << f.sh) - (unsigned long long)d)) / (unsigned long long)d + 1ull);
  return f;
}
__device__ __forceinline__ int fdiv(int n, const FastDiv& f) {
  return (int)((__umulhi(f.mul, (uint32_t)n) + (uint32_t)n) >> f.sh);
}

// ---- cudaLaunchKernelEx with a 1-D thread-block cluster of `cluster` CTAs (no attribute when cluster == 1)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                 int cluster, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = cluster > 1 ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace fidm
