#include "host_common.h"

#include <stdarg.h>
#include <stdio.h>
#include <string.h>

namespace fbkst {

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) !=
          cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

int make_tensor_map(CUtensorMap* out, const void* base, CUtensorMapDataType dtype, int elem_bytes,
                    int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, const uint32_t* elem_strides,
                    CUtensorMapSwizzle swizzle) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error(FBKST_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0)
    return set_error(FBKST_ERR_ARG, "tensor base %p is not 16-byte aligned", base);
  cuuint64_t gdim[5], gstr[5];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = elem_strides ? elem_strides[i] : 1;
    if (i + 1 < rank) {
      gstr[i] = strides_bytes[i];
      if (gstr[i] % 16 != 0)
        return set_error(FBKST_ERR_ARG, "tensor stride %llu B (dim %d) not a multiple of 16",
                         (unsigned long long)gstr[i], i + 1);
    }
  }
  (void)elem_bytes;
  CUresult r = fn(out, dtype, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return set_error(FBKST_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rank %d)",
                     (int)r, rank);
  return FBKST_OK;
}

int make_tensor_map_2d_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols,
                            uint64_t ld, uint32_t box_rows, uint32_t box_cols) {
  uint64_t dims[2] = {cols, rows};
  uint64_t strides[1] = {ld * 2};
  uint32_t box[2] = {box_cols, box_rows};
  return make_tensor_map(out, base, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 2, dims, strides, box,
                         nullptr);
}

int num_sms() {
  static std::atomic<int> cache[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev > 63) return 148;
  int n = cache[dev].load(std::memory_order_relaxed);
  if (n) return n;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
    n = 148;
  cache[dev].store(n, std::memory_order_relaxed);
  return n;
}

}  // namespace fbkst

extern "C" const char* fbkst_last_error(void) { return fbkst::g_err; }
extern "C" int fbkst_abi_version(void) { return 1; }
extern "C" int fbkst_device_ok(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return 0;
  }
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess)
    return 0;
  return major == 10 ? 1 : 0;
}
