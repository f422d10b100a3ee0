// Host-side helpers shared by the C-ABI entry points: error reporting (no exceptions
// cross the ABI) and TMA tensor-map construction through the driver entry point
// (no link-time dependency on libcuda: the symbol is resolved with
// cudaGetDriverEntryPoint at first use).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "../../include/fbkst_b200.h"

namespace fbkst {

// Records `msg` (thread-local) and returns `code`.
int set_error(int code, const char* fmt, ...);

#define FBKST_CHECK_CUDA(expr)                                                              \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess)                                                                  \
      return ::fbkst::set_error(                                                            \
          _e == cudaErrorMemoryAllocation ? FBKST_ERR_OOM : FBKST_ERR_CUDA,                 \
          "%s failed: %s%s", #expr, cudaGetErrorString(_e),                                 \
          _e == cudaErrorMemoryAllocation ? " (CUDA out of memory)" : "");                  \
  } while (0)

#define FBKST_REQUIRE(cond, ...)                                                            \
  do {                                                                                      \
    if (!(cond)) return ::fbkst::set_error(FBKST_ERR_ARG, __VA_ARGS__);                     \
  } while (0)

// rank-N bf16/fp32 tiled tensor map, 128B swizzle.  dims/strides innermost first;
// strides_bytes[i] is the byte stride of dim i+1 (dim 0 is contiguous).
int make_tensor_map(CUtensorMap* out, const void* base, CUtensorMapDataType dtype, int elem_bytes,
                    int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, const uint32_t* elem_strides,
                    CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B);

// 2-D row-major [rows, cols] bf16 matrix with row pitch `ld` elements; box = {box_cols, box_rows}.
int make_tensor_map_2d_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols,
                            uint64_t ld, uint32_t box_rows, uint32_t box_cols);

int num_sms();  // of the CURRENT device (cached per device)

// "already configured on the CURRENT device" flag for one-time per-device setup at a call site
// (cudaFuncSetAttribute is per device; a process may drive several GPUs).  Used as
//   static PerDeviceFlag configured;  if (!configured) { ...; configured = true; }
// Two threads racing on the same device both run the (idempotent) setup before either launches.
class PerDeviceFlag {
 public:
  explicit operator bool() const { return (mask_.load(std::memory_order_acquire) >> dev()) & 1ull; }
  bool operator!() const { return !static_cast<bool>(*this); }
  PerDeviceFlag& operator=(bool v) {
    if (v) mask_.fetch_or(1ull << dev(), std::memory_order_release);
    return *this;
  }

 private:
  static int dev() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d > 63) d = 0;
    return d;
  }
  std::atomic<uint64_t> mask_{0};
};

// conv1 on the tensor pipe (conv1_tcgen05.cu); C is 64 or 128
int conv1_tc_dispatch(const float* x, const float* w, const float* bias, const float* scale,
                      const float* shift, void* y, int B, int T, int F, int C, int T1, int F1, cudaStream_t st);

// Launch `kernel` with programmatic stream serialisation (programmatic dependent launch): the grid
// may be scheduled while the previous kernel of the stream is still draining, runs its prologue
// (barrier init, TMEM allocation, tensor-map prefetch) and blocks in `griddepcontrol.wait` until
// the predecessor has completed and flushed.  Every kernel launched this way MUST execute
// pdl_wait() (ptx.cuh) before its first access to global memory.  Works under stream capture
// (programmatic graph edges).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

}  // namespace fbkst
