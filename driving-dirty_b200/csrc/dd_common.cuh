// Shared helpers for libdd_b200: error text, launch accounting and attributes, dtype load/store.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/dd_b200.h"

namespace dd {

extern thread_local char g_err[512];
extern long long g_launches;

int fail(int code, const char* fmt, ...);
int check_launch(const char* what);  // cudaGetLastError -> return code, counts the launch

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Raises a kernel's dynamic shared-memory limit to `bytes`; reports a failure through fail(), naming `what`.
// Persistent kernels that live on big dynamic shared memory also ask for the maximum shared-memory carveout: an SM changes
// its L1 / shared split only when idle, so a kernel that needs more shared memory than the split chosen for the previous
// one cannot join an SM that the overlapped optimizer update keeps busy (it queued behind the whole update at N > 1).
enum class Carveout { kDefault, kMaxShared };
template <class K>
inline int set_smem(K kernel, size_t bytes, Carveout carveout, const char* what) {
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (carveout == Carveout::kMaxShared)
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return fail((int)e, "%s: cudaFuncSetAttribute(%zu): %s", what, bytes, cudaGetErrorString(e));
  return 0;
}

inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

#define DD_REQUIRE(cond, code, ...) \
  do {                              \
    if (!(cond)) return dd::fail((code), __VA_ARGS__); \
  } while (0)

constexpr int kSMs = 148;  // B200

// ---- activation element access: T = float or __nv_bfloat16, math in fp32 ----
template <typename T> __device__ __forceinline__ float ld(const T* p);
template <> __device__ __forceinline__ float ld<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ld<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}
template <typename T> __device__ __forceinline__ void st(T* p, float v);
template <> __device__ __forceinline__ void st<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void st<__nv_bfloat16>(__nv_bfloat16* p, float v) {
  *p = __float2bfloat16_rn(v);
}

// 8 consecutive elements (32 B of fp32 or 16 B of bf16), pointer aligned accordingly
template <typename T> __device__ __forceinline__ void ld8(const T* p, float (&v)[8]);
template <> __device__ __forceinline__ void ld8<float>(const float* p, float (&v)[8]) {
  float4 a = *reinterpret_cast<const float4*>(p);
  float4 b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
template <> __device__ __forceinline__ void ld8<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[8]) {
  uint4 r = *reinterpret_cast<const uint4*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 f = __bfloat1622float2(h[i]);
    v[2 * i] = f.x; v[2 * i + 1] = f.y;
  }
}
template <typename T> __device__ __forceinline__ void st8(T* p, const float (&v)[8]);
template <> __device__ __forceinline__ void st8<float>(float* p, const float (&v)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
template <> __device__ __forceinline__ void st8<__nv_bfloat16>(__nv_bfloat16* p, const float (&v)[8]) {
  uint4 r;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
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
__device__ __forceinline__ long long warp_sum(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// torchvision ToTensor (data_helper.py:109-114): byte -> float32, divided by 255.  The IEEE division (bit-identical to
// x.float() / 255) is done ONCE per CTA for the 256 possible bytes into a shared-memory table; a division per pixel
// made the raw-byte kernels instruction-bound (the c1 forward + weight gradient pair ran 1.6 ms slower per step).
// Callers look a byte up only after its global load and the loads issued behind it: a look-up at load time makes every
// prefetched load wait for its own round trip (the raw-byte c1 weight gradient ran 0.37 ms against 0.25 for fp32 views).
template <typename TIN> __device__ __forceinline__ float c1_cvt(TIN x, const float* lut);
template <> __device__ __forceinline__ float c1_cvt<float>(float x, const float*) { return x; }
template <> __device__ __forceinline__ float c1_cvt<uint8_t>(uint8_t x, const float* lut) { return lut[x]; }
__device__ __forceinline__ void c1_fill_lut(float* lut) {
  for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = __fdiv_rn((float)i, 255.0f);
}

// mosaic slot j shows dataset view kViewOrder[j] (roadmap_bce_v2.py:58)
__device__ __forceinline__ int view_of_slot(int j) { return j < 3 ? j : 8 - j; }

}  // namespace dd
