// Shared host/device helpers for libhulk_sm100.so.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/hulk_sm100.h"

namespace hk {

// Thread-local last-error text (hk_last_error()).
void set_error(const char* fmt, ...);
int fail(int code, const char* fmt, ...);

// Check the launch that was just enqueued; returns HK_OK or records the CUDA error text.
int check_launch(const char* what);

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline long long ceil_div_ll(long long a, long long b) { return (a + b - 1) / b; }

// Number of SMs of the current device (cached).
int sm_count();

// TMA tensor maps.  Each returns HK_OK, or records "<who>: cuTensorMapEncodeTiled(<what>) failed: <CUresult>" and returns HK_ERR_CUDA.
// bf16 NHWC (n, h, w, c): 64-channel x box_w x box_h boxes, SWIZZLE_128B, L2 promotion 128 B.  step > 1: the box spans step*box_w x
// step*box_h pixels and TMA keeps every step-th (the activation operand of a strided conv).
int tmap_nhwc_bf16(CUtensorMap* m, const void* p, int n, int h, int w, int c, int box_w, int box_h, int step, const char* who,
                   const char* what);
// bf16 K-major (rows, k), row pitch 2k bytes: 64 x box_rows boxes, SWIZZLE_128B, L2 promotion 256 B.
int tmap_kmajor_bf16(CUtensorMap* m, const void* p, long long k, int rows, int box_rows, const char* who, const char* what);
// Any other map: the raw cuTensorMapEncodeTiled arrays (no interleave; out-of-bounds elements read as zero).
int tmap_encode(CUtensorMap* m, CUtensorMapDataType dtype, int rank, const void* p, const cuuint64_t* dims, const cuuint64_t* strides,
                const cuuint32_t* box, const cuuint32_t* estr, CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2, const char* who,
                const char* what);

// Allow Kernel `bytes` of dynamic shared memory on the current device (the attribute is per function and per device).  Sets the
// attribute only when `bytes` exceeds the largest size already set there.
template <auto Kernel>
int opt_in_smem(int bytes, const char* who) {
  static int set_bytes[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  const bool tracked = dev >= 0 && dev < 64;  // beyond the table: set it every time
  if (tracked && set_bytes[dev] >= bytes) return HK_OK;
  const cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return fail(HK_ERR_CUDA, "%s: smem attribute (%d B): %s", who, bytes, cudaGetErrorString(e));
  if (tracked) set_bytes[dev] = bytes;
  return HK_OK;
}

// N tile of the CTA-pair conv kernels.  256 columns amortise the activation tile best, but with few tiles the last wave of the
// persistent grid is mostly idle (batch 4 of 60x80 maps: 75 tiles on 74 CTA pairs = 2 waves for 1.01 waves of work); 128-column tiles
// halve the quantum at ~10 % lower per-tile efficiency.  m_tiles = number of 256-pixel tiles.
inline int pick_block_n_pair(int out_c, long long m_tiles) {
  if (out_c % 256 != 0) return 128;
  const long long clusters = sm_count() / 2;
  const long long t256 = m_tiles * (out_c / 256);
  const double cost256 = (double)ceil_div_ll(t256, clusters);
  const double cost128 = (double)ceil_div_ll(2 * t256, clusters) * 0.55;
  return cost128 < cost256 ? 128 : 256;
}

// Launch with programmatic stream serialization (PDL): the kernel may begin (prologue: barrier init, TMEM allocation, tensor-map
// prefetch) while the previous kernel in the stream drains its last tiles; it MUST execute griddepcontrol.wait before its first
// access to global memory.  HK_PDL=0 falls back to a plain launch.  Works under stream capture (programmatic graph edges).
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

#define HK_REQUIRE(cond, ...)                                  \
  do {                                                         \
    if (!(cond)) return ::hk::fail(HK_ERR_BAD_ARG, __VA_ARGS__); \
  } while (0)

// ---- device helpers ----
__device__ __forceinline__ float bf16_bits_to_float(uint16_t v) { return __uint_as_float(((uint32_t)v) << 16); }

// ToTensor's uint8 / 255 (reference src/dataset.py:16) for operands that are rounded to bf16 right away: for every byte value b,
// bf16_rn(float(b) / 255.0f) == bf16_rn(float(b) * kInv255) (the fp32 results differ by one ulp for 126 of the 256 values, never across
// a bf16 rounding boundary; checked exhaustively, tests/test_host_api.py::test_u8_scale_by_reciprocal_is_exact_in_bf16), so the tensor-core
// stems multiply instead of issuing three IEEE divisions per pixel.  The fp32 correctness mode keeps the division.
constexpr float kInv255 = 1.0f / 255.0f;
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void unpack_bf16x2(uint32_t v, float& lo, float& hi) {
  lo = __uint_as_float(v << 16);
  hi = __uint_as_float(v & 0xffff0000u);
}

template <typename T>
__device__ __forceinline__ float load_as_float(const T* p);
template <>
__device__ __forceinline__ float load_as_float<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float load_as_float<__nv_bfloat16>(const __nv_bfloat16* p) {
  return bf16_bits_to_float(__ldg(reinterpret_cast<const unsigned short*>(p)));
}
template <typename T>
__device__ __forceinline__ void store_from_float(T* p, float v);
template <>
__device__ __forceinline__ void store_from_float<float>(float* p, float v) { *p = v; }
template <>
__device__ __forceinline__ void store_from_float<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

}  // namespace hk
