// Library-level entry points (version, error text, device check) and the host helpers every launcher shares.
#include <stdarg.h>
#include <string.h>

#include "hk_common.cuh"

namespace hk {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(HK_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return HK_OK;
}

int sm_count() {
  static thread_local int cached_dev = -1;
  static thread_local int cached = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached = n;
    cached_dev = dev;
  }
  return cached;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// The driver's cuTensorMapEncodeTiled, looked up once (nullptr when the driver does not provide it).
static EncodeTiledFn get_encode_fn() {
  static const EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool ok = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
                    q == cudaDriverEntryPointSuccess;
    return ok ? reinterpret_cast<EncodeTiledFn>(p) : nullptr;
  }();
  return fn;
}

int tmap_encode(CUtensorMap* m, CUtensorMapDataType dtype, int rank, const void* p, const cuuint64_t* dims, const cuuint64_t* strides,
                const cuuint32_t* box, const cuuint32_t* estr, CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2, const char* who,
                const char* what) {
  const EncodeTiledFn encode = get_encode_fn();
  if (!encode) return fail(HK_ERR_CUDA, "%s: cuTensorMapEncodeTiled entry point not available", who);
  const CUresult r = encode(m, dtype, (cuuint32_t)rank, const_cast<void*>(p), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            swizzle, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(HK_ERR_CUDA, "%s: cuTensorMapEncodeTiled(%s) failed: %d", who, what, (int)r);
  return HK_OK;
}

int tmap_nhwc_bf16(CUtensorMap* m, const void* p, int n, int h, int w, int c, int box_w, int box_h, int step, const char* who,
                   const char* what) {
  const cuuint64_t dims[4] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
  const cuuint64_t strides[3] = {(cuuint64_t)c * 2, (cuuint64_t)w * c * 2, (cuuint64_t)h * w * c * 2};
  const cuuint32_t box[4] = {64, (cuuint32_t)(box_w * step), (cuuint32_t)(box_h * step), 1};
  const cuuint32_t estr[4] = {1, (cuuint32_t)step, (cuuint32_t)step, 1};
  return tmap_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, p, dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, who, what);
}

int tmap_kmajor_bf16(CUtensorMap* m, const void* p, long long k, int rows, int box_rows, const char* who, const char* what) {
  const cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)k * 2};
  const cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return tmap_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, p, dims, strides, box, estr, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, who, what);
}

}  // namespace hk

extern "C" {

int hk_version(void) { return HK_ABI_VERSION; }

const char* hk_last_error(void) { return hk::g_err; }

int hk_check_device(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return hk::fail(HK_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (major != 10 || minor != 0)
    return hk::fail(HK_ERR_UNSUPPORTED_ARCH, "device %d is sm_%d%d; libhulk_sm100 is built for sm_100a only", dev, major, minor);
  return HK_OK;
}

}  // extern "C"
