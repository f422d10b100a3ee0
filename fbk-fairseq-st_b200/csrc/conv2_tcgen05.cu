// conv2 of the subsampling stack (reference: conv_transformer.py:203-214, i=1) as an
// implicit GEMM on tcgen05:  out[(b,t,f), co] = sum_{kh,kw,ci} x[b, 2t-1+kh, 2f-1+kw, ci] * w[co,ci,kh,kw]
//
// No im2col buffer: for each of the 9 taps the A tile (R output rows x F2 output columns x 64
// input channels) is ONE TMA box over the channels-last conv1 output with element strides
// {1,2,2,1}; the box's start coordinate (kw-1, 2*t0+kh-1) goes out of bounds at the borders and
// TMA's zero fill is exactly the conv's zero padding.  K loop = 9 taps x (C/64) channel chunks.
// Operands (conv1 output, weights) and the output are IEEE fp16 (see ptx.cuh idesc_f16_f32).
// Epilogue: +bias -> ReLU -> BatchNorm(eval) affine -> fp16, written channels-last, which is the
// (t, f*C + c) operand layout of the fc3 GEMM (its weight columns are permuted to match).
//
// Warp roles: TMA producer / MMA issuer / TMEM allocator / 4 epilogue warps, persistent.
#include "host_common.h"
#include "ptx.cuh"

namespace fbkst {

struct Conv2Params {
  const float* bias;
  const float* scale;
  const float* shift;
  __nv_bfloat16* out;
  int B, T2, F2, R, tiles_per_utt;
};

template <int C, int STAGES>
__global__ void __launch_bounds__(256, 1)
    conv2_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW,
                 const __grid_constant__ CUtensorMap tmY, Conv2Params p) {
  constexpr int A_BYTES = 128 * 64 * 2;
  constexpr int B_BYTES = C * 64 * 2;
  // C == 64: all nine weight taps (72 KB) stay resident in shared memory for the life of the CTA and a
  // stage holds only the A box (35 % fewer bytes through TMA / L2, two more A stages).  MEASURED: on its
  // own this did not move the kernel (51.2 us at cfg2), nor did unit-stride tap boxes over conv1 output
  // written as four (t1, f1)-parity planes (DESIGN.md finding 15, since removed): the bound was the issue code of the single-lane MMA / TMA warps (see the comment at the
  // warp roles); with that fixed and the epilogue constants in shared memory conv2 runs in 37-40 us.
  constexpr bool WRES = (C == 64);
  constexpr int STAGE_BYTES = A_BYTES + (WRES ? 0 : B_BYTES);
  constexpr int W_BYTES = WRES ? 9 * B_BYTES : 0;
  constexpr int KCH = C / 64;
  constexpr int NUM_KB = 9 * KCH;
  // operand stages + resident taps + 256 B of barriers + 3*C floats of constants, rounded up to 1024
  constexpr int SMEM_MAIN = ((STAGES * STAGE_BYTES + W_BYTES + 256 + 3 * C * 4) + 1023) / 1024 * 1024;
  constexpr uint32_t TMEM_COLS = 2 * C;
  constexpr uint32_t IDESC = idesc_f16_f32(128, C, 0, 0);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // keeps .shared
  uint8_t* sW = smem + STAGES * STAGE_BYTES;  // WRES: [9 taps][C rows][128 B]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sW + W_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* w_full = tempty_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_full + 1);
  // per-channel epilogue constants (bias | BN scale | BN shift), read as broadcast float4 LDS
  float4* sConst = reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(full_bar) + 256);
  // output staging [C/64 halves][128 rows][128 B], 128B-swizzled: one TMA store per tile and half with the
  // box {64, F2, R} of the [B][T2][F2][C] output (rows past T2 are clipped by the map, rows >= R*F2 of the
  // tile are not part of the box), instead of thread-per-row 16-byte stores (32 lines per instruction)
  uint8_t* sOut = smem + SMEM_MAIN;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int num_tiles = p.B * p.tiles_per_utt;
  const uint32_t a_tx = (uint32_t)(p.R * p.F2) * 128u;  // bytes TMA writes for one A box

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmW);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], 4);
    }
    mbar_init(w_full, 1);
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < 3 * C; i += blockDim.x) {
    const float* src = i < C ? p.bias : (i < 2 * C ? p.scale : p.shift);
    reinterpret_cast<float*>(sConst)[i] = __ldg(src + (i % C));
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Both single-issuer roles run in warp-UNIFORM control flow with one elected lane issuing: with
  // `if (lane == 0)` ptxas wraps every UTMALDG / UTCHMMA in a divergence waterfall (ELECT / BRA.U.ANY loop +
  // descriptor rebuild); the MMA warp spent ~60 % of its samples in that issue code and a k-block took ~770
  // cycles for 128 cycles of tensor work (profiles/r01g_ncu_front.txt).
  if (warp == 0) {
    int stage = 0;
    uint32_t phase = 0;
    if (WRES) {
      if (elect_one()) {
        mbar_arrive_expect_tx(w_full, W_BYTES);
        for (int tap = 0; tap < 9; ++tap) tma_load_2d(sW + tap * B_BYTES, &tmW, w_full, 0, tap * C);
      }
      __syncwarp();
    }
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int b = tile / p.tiles_per_utt;
      const int t0 = (tile - b * p.tiles_per_utt) * p.R;
      for (int kb = 0; kb < NUM_KB; ++kb) {
        const int tap = kb / KCH, kc = kb - tap * KCH;
        const int kh = tap / 3, kw = tap - kh * 3;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem + stage * STAGE_BYTES;
        if (elect_one()) {
          mbar_arrive_expect_tx(&full_bar[stage], a_tx + (WRES ? 0 : B_BYTES));
          tma_load_4d(sa, &tmX, &full_bar[stage], kc * 64, kw - 1, 2 * t0 + kh - 1, b);
          if (!WRES) tma_load_2d(sa + A_BYTES, &tmW, &full_bar[stage], kc * 64, tap * C);
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    if (WRES) mbar_wait(w_full, 0);
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * C;
      for (int kb = 0; kb < NUM_KB; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
        const uint64_t adesc = desc_kmajor_sw128(sa);
        const uint64_t bdesc = desc_kmajor_sw128(WRES ? smem_u32(sW) + kb * B_BYTES : sa + A_BYTES);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_bf16_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, IDESC, (kb | k) != 0);
          umma_commit(&empty_bar[stage]);
          if (kb == NUM_KB - 1) umma_commit(&tfull_bar[acc]);  // same thread as the MMAs it tracks
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else if (warp >= 4) {
    const int ew = warp - 4;
    int acc = 0;
    uint32_t acc_phase = 0;
    const int r = ew * 32 + lane;  // tile row == TMEM lane
    uint8_t* srow = sOut + r * 128;
    const bool issuer = (threadIdx.x == 128);
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int b = tile / p.tiles_per_utt;
      const int t0 = (tile - b * p.tiles_per_utt) * p.R;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      if (issuer) tma_store_wait_read<0>();  // the previous tile's store has finished reading the staging tile
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + acc * C;
#pragma unroll 1
      for (int c = 0; c < C / 32; ++c) {
        uint32_t v[32];
        tmem_ld32(taddr + c * 32, v);
        tmem_ld_wait();
        float f[32];
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const float4 bb = sConst[c * 8 + j4], sc = sConst[C / 4 + c * 8 + j4], sh = sConst[C / 2 + c * 8 + j4];
          f[4 * j4 + 0] = fmaf(fmaxf(__uint_as_float(v[4 * j4 + 0]) + bb.x, 0.0f), sc.x, sh.x);
          f[4 * j4 + 1] = fmaf(fmaxf(__uint_as_float(v[4 * j4 + 1]) + bb.y, 0.0f), sc.y, sh.y);
          f[4 * j4 + 2] = fmaf(fmaxf(__uint_as_float(v[4 * j4 + 2]) + bb.z, 0.0f), sc.z, sh.z);
          f[4 * j4 + 3] = fmaf(fmaxf(__uint_as_float(v[4 * j4 + 3]) + bb.w, 0.0f), sc.w, sh.w);
        }
        uint8_t* hrow = srow + (c >> 1) * (128 * 128);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int chunk = (c & 1) * 4 + j;
          *reinterpret_cast<uint4*>(hrow + ((chunk ^ (r & 7)) << 4)) =
              make_uint4(pack_f16x2(f[8 * j], f[8 * j + 1]), pack_f16x2(f[8 * j + 2], f[8 * j + 3]),
                         pack_f16x2(f[8 * j + 4], f[8 * j + 5]), pack_f16x2(f[8 * j + 6], f[8 * j + 7]));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      fence_proxy_async_smem();
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (issuer) {
#pragma unroll
        for (int h = 0; h < C / 64; ++h) tma_store_4d(&tmY, sOut + h * (128 * 128), h * 64, 0, t0, b);
        tma_store_commit();
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (issuer) tma_store_wait<0>();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <int C, int STAGES>
static int launch_conv2(const void* x, const void* w_taps, const Conv2Params& p, int T1, int F1,
                        cudaStream_t stream) {
  constexpr int SMEM_MAIN =
      (((C == 64 ? STAGES * 128 * 64 * 2 + 9 * C * 64 * 2 : STAGES * (128 * 64 * 2 + C * 64 * 2)) + 256 + 3 * C * 4) +
       1023) / 1024 * 1024;
  constexpr int SMEM = SMEM_MAIN + (C / 64) * 128 * 128 /*output staging*/ + 1024 /*alignment slack*/;
  static_assert(SMEM <= 232448, "shared memory budget exceeded");
  auto kern = conv2_kernel<C, STAGES>;
  static PerDeviceFlag configured;
  if (!configured) {
    FBKST_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    configured = true;
  }
  CUtensorMap tmX, tmW;
  int rc;
  {
    uint64_t dims[4] = {(uint64_t)C, (uint64_t)F1, (uint64_t)T1, (uint64_t)p.B};
    uint64_t strides[3] = {(uint64_t)C * 2, (uint64_t)F1 * C * 2, (uint64_t)T1 * F1 * C * 2};
    uint32_t box[4] = {64, (uint32_t)(2 * p.F2), (uint32_t)(2 * p.R), 1};
    uint32_t es[4] = {1, 2, 2, 1};
    rc = make_tensor_map(&tmX, x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 4, dims, strides, box, es);
  }
  if (rc) return rc;
  rc = make_tensor_map_2d_bf16(&tmW, w_taps, (uint64_t)9 * C, (uint64_t)C, (uint64_t)C, C, 64);
  if (rc) return rc;
  CUtensorMap tmY;
  {
    uint64_t dims[4] = {(uint64_t)C, (uint64_t)p.F2, (uint64_t)p.T2, (uint64_t)p.B};
    uint64_t strides[3] = {(uint64_t)C * 2, (uint64_t)p.F2 * C * 2, (uint64_t)p.T2 * p.F2 * C * 2};
    uint32_t box[4] = {64, (uint32_t)p.F2, (uint32_t)p.R, 1};
    rc = make_tensor_map(&tmY, p.out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 4, dims, strides, box, nullptr);
    if (rc) return rc;
  }
  const int tiles = p.B * p.tiles_per_utt;
  const int grid = tiles < num_sms() ? tiles : num_sms();
  kern<<<grid, 256, SMEM, stream>>>(tmX, tmW, tmY, p);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

}  // namespace fbkst

extern "C" int fbkst_conv2_relu_bn(const void* x, const void* w_taps, const float* bias,
                                   const float* bn_scale, const float* bn_shift, void* y, int B,
                                   int T1, int F1, int C, fbkst_stream_t stream) {
  using namespace fbkst;
  FBKST_REQUIRE(x && w_taps && bias && bn_scale && bn_shift && y, "fbkst_conv2_relu_bn: null pointer");
  FBKST_REQUIRE(C == 64 || C == 128, "fbkst_conv2_relu_bn: C must be 64 or 128 (got %d)", C);
  FBKST_REQUIRE(B > 0 && T1 > 0 && F1 > 0, "fbkst_conv2_relu_bn: bad shape");
  Conv2Params p;
  p.bias = bias;
  p.scale = bn_scale;
  p.shift = bn_shift;
  p.out = reinterpret_cast<__nv_bfloat16*>(y);
  p.B = B;
  p.T2 = (T1 + 1) / 2;
  p.F2 = (F1 + 1) / 2;
  FBKST_REQUIRE(p.F2 <= 128, "fbkst_conv2_relu_bn: F2=%d exceeds one 128-row tile", p.F2);
  p.R = 128 / p.F2;
  if (p.R > p.T2) p.R = p.T2;
  p.tiles_per_utt = (p.T2 + p.R - 1) / p.R;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (C == 64) return launch_conv2<64, 8>(x, w_taps, p, T1, F1, st);  // resident weights leave room for 8 A stages
  return launch_conv2<128, 6>(x, w_taps, p, T1, F1, st);
}
