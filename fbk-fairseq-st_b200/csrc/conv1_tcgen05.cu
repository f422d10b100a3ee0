// conv1 of the subsampling stack (reference: conv_transformer.py:203-214, i=0: Conv2d(1, C, 3, stride 2,
// padding 1) -> ReLU -> BatchNorm2d(eval)) on the tensor pipe.
//
// Cin = 1, so the implicit GEMM has K = 9: far too little work to be tensor-bound -- the kernel's job is
// to WRITE 2*C bytes per output pixel (cfg2: 123 MB) at HBM speed, and the SIMT version this replaced
// (since removed: 72 FMAs + epilogue per pixel and 8-channel group, 128 registers) spent 65 us issuing
// instructions for a 19 us write.  Here one tile = 128 consecutive output pixels (the channels-last output
// is one contiguous [pixels, C] matrix):
//   build     thread <-> pixel: 9 predicated loads (zero outside the image = the conv padding), fp16,
//             two 16-byte chunks into a K-major 128B-swizzled A tile (K padded 9 -> 16, ONE UMMA k-step)
//   MMA       one tcgen05.mma M128 x N=C x K16 against the weight tile (built once per CTA), fp32 in TMEM
//   epilogue  thread <-> TMEM lane <-> pixel: +bias -> ReLU -> BatchNorm affine -> fp16 -> swizzled smem
//             row -> one TMA store per warp (32 pixels x 128 B), rows past the end clipped by the map
// Small CTAs (160 threads, ~42 KB smem, C TMEM columns), as many per SM as fit: while one CTA waits for
// its loads or its MMA the others build / drain.  Inputs, weights and the output are IEEE fp16 (saturating
// conversions; accumulation stays fp32): the front end runs in fp16, not bf16 -- see ptx.cuh idesc_f16_f32.
#include "host_common.h"
#include "ptx.cuh"

namespace fbkst {

constexpr int C1_THREADS = 160;  // warp 0: TMEM allocator + MMA issuer; warps 1-4: build + epilogue

template <int C>
__global__ void __launch_bounds__(C1_THREADS, 4)
    conv1_tc_kernel(const __grid_constant__ CUtensorMap tmY, const float* __restrict__ x,
                    const float* __restrict__ w, const float* __restrict__ bias,
                    const float* __restrict__ scale, const float* __restrict__ shift, int T, int F,
                    int T1, int F1, int n_pix) {
  constexpr uint32_t IDESC = idesc_f16_f32(128, C, 0, 0);
  constexpr int HALVES = C / 64;                 // 64-column (128-byte) output pieces per pixel
  constexpr int OUT_WARP_BYTES = HALVES * 4096;  // [half][32 rows][128 B] per epilogue warp

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;                         // [128 rows][128 B], only the first k-step (32 B/row) is used
  uint8_t* sW = sA + 128 * 128;               // [C rows][128 B]
  uint8_t* sOut = sW + C * 128;               // 4 x OUT_WARP_BYTES
  float4* sConst = reinterpret_cast<float4*>(sOut + 4 * OUT_WARP_BYTES);  // bias | scale | shift, C floats each
  uint64_t* a_full = reinterpret_cast<uint64_t*>(sConst + 3 * C / 4);
  uint64_t* mma_done = a_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_done + 1);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int n_tiles = (n_pix + 127) / 128;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmY);
    mbar_init(a_full, 128);
    mbar_init(mma_done, 1);
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_slot, C);
    tmem_relinquish();
  }
  // weight tile: row n = output channel, K-major, k = kh*3 + kw in the first 16-element k-step
  for (int n = threadIdx.x; n < C; n += C1_THREADS) {
    float wv[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) wv[k] = __ldg(w + n * 9 + k);
    uint8_t* rowp = sW + n * 128;
    *reinterpret_cast<uint4*>(rowp + ((0 ^ (n & 7)) << 4)) =
        make_uint4(pack_f16x2(wv[0], wv[1]), pack_f16x2(wv[2], wv[3]), pack_f16x2(wv[4], wv[5]),
                   pack_f16x2(wv[6], wv[7]));
    *reinterpret_cast<uint4*>(rowp + ((1 ^ (n & 7)) << 4)) = make_uint4(pack_f16x2(wv[8], 0.0f), 0u, 0u, 0u);
  }
  for (int i = threadIdx.x; i < 3 * C; i += C1_THREADS) {
    const float* src = i < C ? bias : (i < 2 * C ? scale : shift);
    reinterpret_cast<float*>(sConst)[i] = __ldg(src + (i % C));
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ MMA issuer
    const uint64_t adesc = desc_kmajor_sw128(smem_u32(sA));
    const uint64_t bdesc = desc_kmajor_sw128(smem_u32(sW));
    uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ph ^= 1) {
      mbar_wait(a_full, ph);  // A tile written, and every thread has read the previous accumulator
      tc_fence_after();
      if (elect_one()) {
        umma_bf16_ss(tmem_base, adesc, bdesc, IDESC, 0);
        umma_commit(mma_done);
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------------------------------------ build + epilogue
    const int q = warp & 3;            // TMEM lane quarter of this warp
    const int row = q * 32 + lane;     // tile row == TMEM lane == pixel
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    uint8_t* a_row = sA + row * 128;
    const int sw = row & 7;
    uint8_t* out_warp = sOut + q * OUT_WARP_BYTES;
    const int ppu = T1 * F1;  // pixels per utterance
    uint32_t ph = 0;
    float in[9];
    auto load_taps = [&](int tile) {  // the 9 taps of this thread's pixel of `tile` (zero outside the image)
      const int p = tile * 128 + row;
#pragma unroll
      for (int k = 0; k < 9; ++k) in[k] = 0.0f;
      if (tile < n_tiles && p < n_pix) {
        const int b = p / ppu;
        const int rem = p - b * ppu;
        const int t1 = rem / F1;
        const int f1 = rem - t1 * F1;
        const float* xb = x + (size_t)b * T * F;
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
          const int t = 2 * t1 - 1 + kh;
          if (t >= 0 && t < T) {
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) {
              const int f = 2 * f1 - 1 + kw;
              if (f >= 0 && f < F) in[kh * 3 + kw] = __ldg(xb + (size_t)t * F + f);
            }
          }
        }
      }
    };
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ph ^= 1) {
      // ---- build.  (Fetching the NEXT tile's taps here, under this tile's MMA and epilogue, was measured
      // slower: 57 vs 41 us at cfg2 -- the other CTAs of the SM already cover the load latency.)
      load_taps(tile);
      *reinterpret_cast<uint4*>(a_row + ((0 ^ sw) << 4)) =
          make_uint4(pack_f16x2(in[0], in[1]), pack_f16x2(in[2], in[3]), pack_f16x2(in[4], in[5]),
                     pack_f16x2(in[6], in[7]));
      *reinterpret_cast<uint4*>(a_row + ((1 ^ sw) << 4)) = make_uint4(pack_f16x2(in[8], 0.0f), 0u, 0u, 0u);
      fence_proxy_async_smem();
      tc_fence_before();  // orders the previous tile's TMEM reads before the MMA this arrival releases
      mbar_arrive(a_full);
      // the previous tile's TMA store must have finished READING this warp's staging rows
      if (lane == 0) tma_store_wait_read<0>();
      __syncwarp();
      mbar_wait(mma_done, ph);
      tc_fence_after();
      // ---- epilogue: +bias -> ReLU -> BN affine -> fp16, 32 columns at a time
#pragma unroll
      for (int c32 = 0; c32 < C / 32; ++c32) {
        uint32_t v[32];
        tmem_ld32(taddr + c32 * 32, v);
        tmem_ld_wait();
        uint8_t* orow = out_warp + (c32 >> 1) * 4096 + lane * 128;
#pragma unroll
        for (int j = 0; j < 4; ++j) {  // 8 columns -> one 16-byte chunk
          float o[8];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int c4 = c32 * 8 + j * 2 + h;  // float4 index into the channel constants
            const float4 bb = sConst[c4], sc = sConst[C / 4 + c4], sh = sConst[2 * C / 4 + c4];
            const float a0 = fmaxf(__uint_as_float(v[j * 8 + h * 4 + 0]) + bb.x, 0.0f);
            const float a1 = fmaxf(__uint_as_float(v[j * 8 + h * 4 + 1]) + bb.y, 0.0f);
            const float a2 = fmaxf(__uint_as_float(v[j * 8 + h * 4 + 2]) + bb.z, 0.0f);
            const float a3 = fmaxf(__uint_as_float(v[j * 8 + h * 4 + 3]) + bb.w, 0.0f);
            o[h * 4 + 0] = fmaf(a0, sc.x, sh.x);
            o[h * 4 + 1] = fmaf(a1, sc.y, sh.y);
            o[h * 4 + 2] = fmaf(a2, sc.z, sh.z);
            o[h * 4 + 3] = fmaf(a3, sc.w, sh.w);
          }
          const int chunk = (c32 & 1) * 4 + j;  // 16-byte chunk inside the 128-byte half row
          *reinterpret_cast<uint4*>(orow + ((chunk ^ (lane & 7)) << 4)) =
              make_uint4(pack_f16x2(o[0], o[1]), pack_f16x2(o[2], o[3]), pack_f16x2(o[4], o[5]),
                         pack_f16x2(o[6], o[7]));
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
#pragma unroll
        for (int h = 0; h < HALVES; ++h) tma_store_2d(&tmY, out_warp + h * 4096, h * 64, tile * 128 + q * 32);
        tma_store_commit();
      }
    }
    if (lane == 0) tma_store_wait<0>();  // global writes complete before the CTA exits
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C);
  }
}

template <int C>
static int launch_conv1_tc(const float* x, const float* w, const float* bias, const float* scale,
                           const float* shift, void* y, int B, int T, int F, int T1, int F1, cudaStream_t st) {
  constexpr int SMEM = 128 * 128 + C * 128 + 4 * (C / 64) * 4096 + 3 * C * 4 + 64 + 1024;
  auto kern = conv1_tc_kernel<C>;
  static PerDeviceFlag configured;
  if (!configured) {
    // (no shared-memory carve-out preference: the driver default and 100 % measure the same, 41 us)
    FBKST_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    configured = true;
  }
  const long long n_pix = (long long)B * T1 * F1;
  FBKST_REQUIRE(n_pix < (1ll << 31), "fbkst_conv1_relu_bn: too many pixels");
  CUtensorMap tmY;
  uint64_t dims[2] = {(uint64_t)C, (uint64_t)n_pix};
  uint64_t strides[1] = {(uint64_t)C * 2};
  uint32_t box[2] = {64u, 32u};
  int rc = make_tensor_map(&tmY, y, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 2, dims, strides, box, nullptr);
  if (rc) return rc;
  const int n_tiles = (int)((n_pix + 127) / 128);
  // CTAs per SM by hand: 43 KB (C=64) / 67 KB (C=128) of smem, 80-85 registers x 160 threads and C TMEM
  // columns give 4 / 3.  cudaOccupancyMaxActiveBlocksPerMultiprocessor answers 1 for this kernel (it
  // appears to charge a tcgen05.alloc-ing kernel the whole TMEM), which halves the throughput: measured
  // 3 / 4 / 5 / 6 CTAs per SM -> 49 / 41 / 53 / 49 us at cfg2, 1 -> 86 us.
  const int per_sm = (C == 64) ? 4 : 3;
  int grid = num_sms() * per_sm;
  if (grid > n_tiles) grid = n_tiles;
  kern<<<grid, C1_THREADS, SMEM, st>>>(tmY, x, w, bias, scale, shift, T, F, T1, F1, (int)n_pix);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

int conv1_tc_dispatch(const float* x, const float* w, const float* bias, const float* scale,
                      const float* shift, void* y, int B, int T, int F, int C, int T1, int F1, cudaStream_t st) {
  if (C == 64) return launch_conv1_tc<64>(x, w, bias, scale, shift, y, B, T, F, T1, F1, st);
  return launch_conv1_tc<128>(x, w, bias, scale, shift, y, B, T, F, T1, F1, st);
}

}  // namespace fbkst
