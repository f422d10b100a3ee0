// out = epilogue(A @ W^T): persistent, warp-specialised tcgen05 GEMM for sm_100a.
//
//   warp 0      TMA producer      (one elected lane; A and W tiles, 128B swizzle)
//   warp 1      MMA issuer        (one lane; tcgen05.mma kind::f16, fp32 accumulators in TMEM)
//   warp 2      TMEM allocator
//   warps 4-7   epilogue          (tcgen05.ld -> bias/ReLU/residual/pos-emb -> global)
//
// Tile 128 x BN x 64, STAGES-deep smem ring, two TMEM accumulator stages so that the epilogue
// of tile i overlaps the main loop of tile i+1.  It serves the row-remap / position-embedding
// epilogues; fbkst_linear_bf16 sends every other nn.Linear of the reference path
// (conv_transformer.py:227,279; local_attention.py:178,141; transformer_layer.py:131-133) to the
// CTA-pair kernel of gemm2_tcgen05.cu.
#include "host_common.h"
#include "ptx.cuh"

namespace fbkst {

// gemm2_tcgen05.cu: CTA-pair (cta_group::2) kernel for the plain / residual epilogues
int linear_pair_dispatch(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                         const float* resid, int64_t ldr, void* out, int64_t ldo, int M, int N, int K,
                         int relu, int out_f32, const int* m_limit, int m_limit_mult,
                         const float* stats_in, float ln_eps, void* out_bf16, int64_t ldob,
                         float* stats_out, int ab_f16, cudaStream_t stream);

struct EpiParams {
  const float* bias;
  const float* resid;
  long long ldr;
  void* out;
  long long ldo;
  const int* lengths;
  int flags;
  int remap_inner;
  int remap_outer;
};

constexpr int BM = 128;
constexpr int BK = 64;

// One thread owns one output row and 32 consecutive columns starting at col0.
__device__ __forceinline__ void epilogue_store(const EpiParams& ep, const uint32_t (&v)[32],
                                               int row, int col0, int N) {
  float f[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
  const bool full = (col0 + 32 <= N);
  if (ep.bias != nullptr) {
    if (full) {
      const float4* bp = reinterpret_cast<const float4*>(ep.bias + col0);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float4 b = __ldg(bp + j);
        f[4 * j + 0] += b.x;
        f[4 * j + 1] += b.y;
        f[4 * j + 2] += b.z;
        f[4 * j + 3] += b.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (col0 + j < N) f[j] += __ldg(ep.bias + col0 + j);
    }
  }
  if (ep.flags & FBKST_EPI_RELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.0f);
  }
  long long orow = row;
  int rb = 0, rt = 0;
  if (ep.flags & (FBKST_EPI_ROW_REMAP | FBKST_EPI_POSEMB)) {
    rb = row / ep.remap_inner;
    rt = row - rb * ep.remap_inner;
    if (ep.flags & FBKST_EPI_ROW_REMAP) orow = (long long)rt * ep.remap_outer + rb;
  }
  if (ep.resid != nullptr) {
    long long rrow = row;
    if (ep.flags & FBKST_EPI_POSEMB) rrow = (rt < __ldg(ep.lengths + rb)) ? (rt + 1) : 0;
    const float* rp = ep.resid + rrow * ep.ldr + col0;
    if (full) {
      const float4* r4 = reinterpret_cast<const float4*>(rp);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float4 r = __ldg(r4 + j);
        f[4 * j + 0] += r.x;
        f[4 * j + 1] += r.y;
        f[4 * j + 2] += r.z;
        f[4 * j + 3] += r.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (col0 + j < N) f[j] += __ldg(rp + j);
    }
  }
  if (ep.flags & FBKST_EPI_OUT_F32) {
    float* op = reinterpret_cast<float*>(ep.out) + orow * ep.ldo + col0;
    if (full) {
      float4* o4 = reinterpret_cast<float4*>(op);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        o4[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (col0 + j < N) op[j] = f[j];
    }
  } else {
    __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(ep.out) + orow * ep.ldo + col0;
    if (full) {
      uint4* o4 = reinterpret_cast<uint4*>(op);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        o4[j] = make_uint4(pack_bf16x2(f[8 * j], f[8 * j + 1]), pack_bf16x2(f[8 * j + 2], f[8 * j + 3]),
                           pack_bf16x2(f[8 * j + 4], f[8 * j + 5]),
                           pack_bf16x2(f[8 * j + 6], f[8 * j + 7]));
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (col0 + j < N) op[j] = __float2bfloat16_rn(f[j]);
    }
  }
}

template <int BN, int STAGES>
__global__ void __launch_bounds__(256, 1)
    gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmA,
                     const __grid_constant__ CUtensorMap tmB, int M, int N, int K, EpiParams ep) {
  constexpr int A_BYTES = BM * BK * 2;
  constexpr int B_BYTES = BN * BK * 2;
  constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr uint32_t TMEM_COLS = 2 * BN;
  constexpr uint32_t IDESC = idesc_bf16_f32(BM, BN, 0, 0);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // keeps .shared
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const int num_n = (N + BN - 1) / BN;
  const int num_m = (M + BM - 1) / BM;
  const int num_tiles = num_m * num_n;
  const int num_kb = (K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
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
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_blk = tile / num_n, n_blk = tile - m_blk * num_n;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], STAGE_BYTES);
          uint8_t* sa = smem + stage * STAGE_BYTES;
          tma_load_2d(sa, &tmA, &full_bar[stage], kb * BK, m_blk * BM);
          tma_load_2d(sa + A_BYTES, &tmB, &full_bar[stage], kb * BK, n_blk * BN);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const uint64_t adesc = desc_kmajor_sw128(sa);
          const uint64_t bdesc = desc_kmajor_sw128(sa + A_BYTES);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            umma_bf16_ss(d_tmem, adesc + 2 * k, bdesc + 2 * k, IDESC, (kb | k) != 0);
          umma_commit(&empty_bar[stage]);
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit(&tfull_bar[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if (warp >= 4) {
    const int ew = warp - 4;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m_blk = tile / num_n, n_blk = tile - m_blk * num_n;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const int row = m_blk * BM + ew * 32 + lane;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + acc * BN;
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        const int col0 = n_blk * BN + c * 32;
        if (col0 >= N) break;  // warp-uniform
        uint32_t v[32];
        tmem_ld32(taddr + c * 32, v);
        tmem_ld_wait();
        if (row < M) epilogue_store(ep, v, row, col0, N);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <int BN, int STAGES>
static int launch_gemm(const void* A, int64_t lda, const void* W, int64_t ldw, int M, int N, int K,
                       const EpiParams& ep, cudaStream_t stream) {
  constexpr int SMEM = STAGES * (BM * BK * 2 + BN * BK * 2) + 1024 + 256;
  static PerDeviceFlag configured;
  auto kern = gemm_bf16_kernel<BN, STAGES>;
  if (!configured) {
    FBKST_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    configured = true;
  }
  CUtensorMap tmA, tmB;
  int rc = make_tensor_map_2d_bf16(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda, BM, BK);
  if (rc) return rc;
  rc = make_tensor_map_2d_bf16(&tmB, W, (uint64_t)N, (uint64_t)K, (uint64_t)ldw, BN, BK);
  if (rc) return rc;
  const int tiles = ((M + BM - 1) / BM) * ((N + BN - 1) / BN);
  const int grid = tiles < num_sms() ? tiles : num_sms();
  kern<<<grid, 256, SMEM, stream>>>(tmA, tmB, M, N, K, ep);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

}  // namespace fbkst

extern "C" int fbkst_linear_bf16(const void* A, int64_t lda, const void* W, int64_t ldw,
                                 const float* bias, const float* residual, int64_t ldr, void* out,
                                 int64_t ldo, int M, int N, int K, int flags, int remap_inner,
                                 int remap_outer, const int32_t* lengths, const int32_t* m_limit,
                                 int m_limit_mult, fbkst_stream_t stream) {
  using namespace fbkst;
  FBKST_REQUIRE(A && W && out, "fbkst_linear_bf16: null operand");
  FBKST_REQUIRE(M > 0 && N > 0 && K > 0, "fbkst_linear_bf16: empty problem M=%d N=%d K=%d", M, N, K);
  FBKST_REQUIRE(K % 8 == 0 && lda % 8 == 0 && ldw % 8 == 0,
                "fbkst_linear_bf16: K, lda, ldw must be multiples of 8 (K=%d lda=%lld ldw=%lld)", K,
                (long long)lda, (long long)ldw);
  FBKST_REQUIRE(ldo % 8 == 0, "fbkst_linear_bf16: ldo must be a multiple of 8 (got %lld)",
                (long long)ldo);
  FBKST_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "fbkst_linear_bf16: out must be 16-byte aligned");
  FBKST_REQUIRE(residual == nullptr || ldr % 4 == 0, "fbkst_linear_bf16: ldr must be a multiple of 4");
  if (flags & (FBKST_EPI_ROW_REMAP | FBKST_EPI_POSEMB))
    FBKST_REQUIRE(remap_inner > 0 && remap_outer > 0, "fbkst_linear_bf16: remap dims required");
  if (flags & FBKST_EPI_POSEMB)
    FBKST_REQUIRE(lengths && residual, "fbkst_linear_bf16: POSEMB needs lengths and a table");
  EpiParams ep;
  ep.bias = bias;
  ep.resid = residual;
  ep.ldr = ldr;
  ep.out = out;
  ep.ldo = ldo;
  ep.lengths = lengths;
  ep.flags = flags;
  ep.remap_inner = remap_inner;
  ep.remap_outer = remap_outer;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (flags & (FBKST_EPI_ROW_REMAP | FBKST_EPI_POSEMB)) {  // row-remapping epilogue: direct stores
    FBKST_REQUIRE(!(flags & FBKST_EPI_AB_F16), "fbkst_linear_bf16: fp16 operands need the CTA-pair kernel");
    FBKST_REQUIRE(m_limit == nullptr, "fbkst_linear_bf16: m_limit is not supported with the row-remap epilogues");
    if (N % 256 == 0 || N > 1024) return launch_gemm<256, 4>(A, lda, W, ldw, M, N, K, ep, st);
    return launch_gemm<128, 6>(A, lda, W, ldw, M, N, K, ep, st);
  }
  const int relu = (flags & FBKST_EPI_RELU) ? 1 : 0;
  if (residual != nullptr)
    FBKST_REQUIRE(flags & FBKST_EPI_OUT_F32, "fbkst_linear_bf16: a residual requires fp32 output");
  return linear_pair_dispatch(A, lda, W, ldw, bias, residual, ldr, out, ldo, M, N, K, relu,
                              (flags & FBKST_EPI_OUT_F32) ? 1 : 0, m_limit, m_limit_mult, nullptr, 0.f, nullptr, 0,
                              nullptr, (flags & FBKST_EPI_AB_F16) ? 1 : 0, st);
}

extern "C" int fbkst_linear_ln_bf16(const void* A, int64_t lda, const void* W, int64_t ldw,
                                    const float* bias, const float* residual, int64_t ldr, void* out,
                                    int64_t ldo, int M, int N, int K, int flags,
                                    const float* row_stats_in, float ln_eps, void* out_bf16,
                                    int64_t ldob, float* row_stats_out, const int32_t* m_limit,
                                    int m_limit_mult, fbkst_stream_t stream) {
  using namespace fbkst;
  FBKST_REQUIRE(A && W && out, "fbkst_linear_ln_bf16: null operand");
  FBKST_REQUIRE(M > 0 && N > 0 && K > 0, "fbkst_linear_ln_bf16: empty problem M=%d N=%d K=%d", M, N, K);
  FBKST_REQUIRE(K % 8 == 0 && lda % 8 == 0 && ldw % 8 == 0 && ldo % 8 == 0,
                "fbkst_linear_ln_bf16: K, lda, ldw, ldo must be multiples of 8");
  FBKST_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "fbkst_linear_ln_bf16: out must be 16-byte aligned");
  FBKST_REQUIRE(!(flags & (FBKST_EPI_ROW_REMAP | FBKST_EPI_POSEMB)),
                "fbkst_linear_ln_bf16: row remap / position epilogues are not available here");
  if (residual != nullptr)
    FBKST_REQUIRE((flags & FBKST_EPI_OUT_F32) && ldr % 4 == 0,
                  "fbkst_linear_ln_bf16: a residual requires fp32 output and ldr %% 4 == 0");
  FBKST_REQUIRE((out_bf16 == nullptr) == (row_stats_out == nullptr),
                "fbkst_linear_ln_bf16: out_bf16 and row_stats_out come together");
  if (row_stats_out != nullptr) {
    FBKST_REQUIRE(residual != nullptr, "fbkst_linear_ln_bf16: row statistics need the residual epilogue");
    FBKST_REQUIRE(N % 32 == 0 && ldob % 8 == 0 && (reinterpret_cast<uintptr_t>(out_bf16) & 15) == 0,
                  "fbkst_linear_ln_bf16: N %% 32, ldob %% 8 and 16-byte alignment required (N=%d)", N);
  }
  if (row_stats_in != nullptr)
    FBKST_REQUIRE(residual == nullptr, "fbkst_linear_ln_bf16: row_stats_in applies to the plain epilogue");
  return linear_pair_dispatch(A, lda, W, ldw, bias, residual, ldr, out, ldo, M, N, K,
                              (flags & FBKST_EPI_RELU) ? 1 : 0, (flags & FBKST_EPI_OUT_F32) ? 1 : 0, m_limit,
                              m_limit_mult, row_stats_in, ln_eps, out_bf16, ldob, row_stats_out,
                              (flags & FBKST_EPI_AB_F16) ? 1 : 0, reinterpret_cast<cudaStream_t>(stream));
}
