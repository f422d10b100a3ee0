// fp32-accurate inference path (DESIGN section F): split-TF32 ("3xTF32") tensor-core kernels for sm_100a.
//
// Every fp32 operand x is split as x = hi + lo with hi = tf32_rna(x) and lo = tf32_rna(x - hi), and a product
// a.b is computed as hi(a).hi(b) + hi(a).lo(b) + lo(a).hi(b) into ONE fp32 accumulator in tensor memory
// (tcgen05.mma kind::tf32, K = 8 per instruction).  The dropped lo.lo term and the rounding of lo leave about
// 21 significant bits per operand, against 11 for plain TF32 (scripts/precision_budget_probe.py).  The tensor
// core truncates an fp32 operand to TF32, so hi must be rounded explicitly (cvt.rna.tf32.f32).
//
// The split happens in shared memory, inside the kernels: activations and weights stay plain fp32 in HBM and
// no other module knows the hi / lo format.
//
//   fbkst_linear_tf32x3      y = A W^T (+ bias, ReLU, per-column affine, fp32 residual), device row limit
//   fbkst_attention_tf32x3   softmax(Q K^T - penalty, key padding) V, fp32 softmax, two exact passes
//   fbkst_conv1_relu_bn_f32  first subsampling convolution (K = 9, SIMT: bound by its output bytes)
//   fbkst_conv2_im2col_f32   the second convolution's patches, for fbkst_linear_tf32x3
#include <math.h>

#include "host_common.h"
#include "ptx.cuh"

namespace fbkst {

// ------------------------------------------------------------------------------------ split helpers
__device__ __forceinline__ float tf32_rna(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  hi = tf32_rna(x);
  lo = tf32_rna(x - hi);
}
__device__ __forceinline__ void split4(const float4& x, float4& hi, float4& lo) {
  split_tf32(x.x, hi.x, lo.x);
  split_tf32(x.y, hi.y, lo.y);
  split_tf32(x.z, hi.z, lo.z);
  split_tf32(x.w, hi.w, lo.w);
}

// Instruction descriptor, kind::tf32: D fp32 (bits 4-5 = 1), A and B format TF32 (bits 7-9 and 10-12 = 2),
// both K-major, N >> 3 at bit 17, M >> 4 at bit 24 (PTX ISA, tcgen05 instruction descriptor).
__host__ __device__ constexpr uint32_t idesc_tf32_f32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void umma_tf32_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// D (+)= Ahi.Bhi + Ahi.Blo + Alo.Bhi for one K = 8 step (descriptors already advanced to the step)
__device__ __forceinline__ void umma_tf32x3(uint32_t d_tmem, uint64_t a_hi, uint64_t a_lo, uint64_t b_hi,
                                            uint64_t b_lo, uint32_t idesc, uint32_t accumulate) {
  umma_tf32_ss(d_tmem, a_lo, b_hi, idesc, accumulate);
  umma_tf32_ss(d_tmem, a_hi, b_lo, idesc, 1u);
  umma_tf32_ss(d_tmem, a_hi, b_hi, idesc, 1u);
}

// =================================================================================== GEMM
//   warp 0      TMA producer   (fp32 tiles 128 x 32 / BN x 32, one 128-byte swizzle atom per row)
//   warp 1      MMA issuer     (3 x 4 tcgen05.mma kind::tf32 per stage)
//   warp 2      TMEM allocator
//   warps 4-7   splitters      (raw fp32 -> hi in place, lo into the stage's second half; same swizzled offsets)
//   warps 8-11  epilogue       (TMEM -> bias / ReLU / affine / residual -> fp32 global)
// Two TMEM accumulator stages: the epilogue of tile i overlaps the main loop of tile i + 1.
constexpr int X3_BM = 128;
constexpr int X3_BN = 128;
constexpr int X3_BK = 32;
constexpr int X3_STAGES = 3;
constexpr int X3_A_BYTES = X3_BM * X3_BK * 4;         // 16 KB
constexpr int X3_B_BYTES = X3_BN * X3_BK * 4;         // 16 KB
constexpr int X3_RAW_BYTES = X3_A_BYTES + X3_B_BYTES;  // raw tile, split in place into hi
constexpr int X3_STAGE_BYTES = 2 * X3_RAW_BYTES;       // hi | lo
constexpr int X3_SMEM = X3_STAGES * X3_STAGE_BYTES + 1024 + 256;

struct X3Epi {
  const float* bias;
  const float* col_scale;  // y = y * col_scale[n] + col_shift[n] after the ReLU (eval BatchNorm), or NULL
  const float* col_shift;
  const float* resid;
  long long ldr;
  float* out;
  long long ldo;
  int relu;
};

__global__ void __launch_bounds__(384, 1)
    gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, int M,
                       int N, int K, const int* __restrict__ m_limit, int m_limit_mult, X3Epi ep) {
  constexpr uint32_t TMEM_COLS = 2 * X3_BN;
  constexpr uint32_t IDESC = idesc_tf32_f32(X3_BM, X3_BN);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + X3_STAGES * X3_STAGE_BYTES);
  uint64_t* split_bar = full_bar + X3_STAGES;
  uint64_t* empty_bar = split_bar + X3_STAGES;
  uint64_t* tfull_bar = empty_bar + X3_STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  if (m_limit != nullptr) M = min(M, __ldg(m_limit) * m_limit_mult);  // rows beyond are neither read nor written
  const int num_n = (N + X3_BN - 1) / X3_BN;
  const int num_m = (M + X3_BM - 1) / X3_BM;
  const int num_tiles = num_m * num_n;
  const int num_kb = (K + X3_BK - 1) / X3_BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < X3_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&split_bar[s], 4);
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
          mbar_arrive_expect_tx(&full_bar[stage], X3_RAW_BYTES);
          uint8_t* sa = smem + stage * X3_STAGE_BYTES;
          tma_load_2d(sa, &tmA, &full_bar[stage], kb * X3_BK, m_blk * X3_BM);
          tma_load_2d(sa + X3_A_BYTES, &tmB, &full_bar[stage], kb * X3_BK, n_blk * X3_BN);
          if (++stage == X3_STAGES) {
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
        const uint32_t d_tmem = tmem_base + acc * X3_BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&split_bar[stage], phase);
          tc_fence_after();
          const uint32_t s0 = smem_u32(smem + stage * X3_STAGE_BYTES);
          const uint64_t a_hi = desc_kmajor_sw128(s0), b_hi = desc_kmajor_sw128(s0 + X3_A_BYTES);
          const uint64_t a_lo = desc_kmajor_sw128(s0 + X3_RAW_BYTES),
                         b_lo = desc_kmajor_sw128(s0 + X3_RAW_BYTES + X3_A_BYTES);
#pragma unroll
          for (int k = 0; k < X3_BK / 8; ++k)  // 8 tf32 = 32 bytes = 2 descriptor units
            umma_tf32x3(d_tmem, a_hi + 2 * k, a_lo + 2 * k, b_hi + 2 * k, b_lo + 2 * k, IDESC, (kb | k) != 0);
          umma_commit(&empty_bar[stage]);
          if (++stage == X3_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit(&tfull_bar[acc]);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if (warp >= 4 && warp < 8) {
    const int t = threadIdx.x - 128;  // 0..127
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        float4* raw = reinterpret_cast<float4*>(smem + stage * X3_STAGE_BYTES);
        float4* lo = reinterpret_cast<float4*>(smem + stage * X3_STAGE_BYTES + X3_RAW_BYTES);
#pragma unroll 4
        for (int i = t; i < X3_RAW_BYTES / 16; i += 128) {
          float4 h, l;
          split4(raw[i], h, l);
          raw[i] = h;
          lo[i] = l;
        }
        fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive(&split_bar[stage]);
        if (++stage == X3_STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp >= 8) {
    const int q = warp & 3;  // TMEM lane quarter (warp % 4 selects the lanes a warp may access)
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m_blk = tile / num_n, n_blk = tile - m_blk * num_n;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const int row = m_blk * X3_BM + q * 32 + lane;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * X3_BN;
#pragma unroll 1
      for (int c = 0; c < X3_BN / 32; ++c) {
        const int col0 = n_blk * X3_BN + c * 32;
        if (col0 >= N) break;  // warp-uniform
        uint32_t v[32];
        tmem_ld32(taddr + c * 32, v);
        tmem_ld_wait();
        if (row < M) {
          float f[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
          const int nv = min(32, N - col0);
          if (ep.bias != nullptr) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j < nv) f[j] += __ldg(ep.bias + col0 + j);
          }
          if (ep.relu) {
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.0f);
          }
          if (ep.col_scale != nullptr) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j < nv) f[j] = fmaf(f[j], __ldg(ep.col_scale + col0 + j), __ldg(ep.col_shift + col0 + j));
          }
          if (ep.resid != nullptr) {
            const float* rp = ep.resid + (long long)row * ep.ldr + col0;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j < nv) f[j] += rp[j];
          }
          float* op = ep.out + (long long)row * ep.ldo + col0;
          if (nv == 32 && ((reinterpret_cast<uintptr_t>(op) & 15) == 0)) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
              reinterpret_cast<float4*>(op)[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j < nv) op[j] = f[j];
          }
        }
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

static int make_map_f32_2d(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                           uint32_t box_rows) {
  uint64_t dims[2] = {cols, rows};
  uint64_t strides[1] = {ld * 4};
  uint32_t box[2] = {32u, box_rows};
  return make_tensor_map(m, base, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, 2, dims, strides, box, nullptr);
}

// =================================================================================== attention
// One CTA (128 threads, one query row per thread == TMEM lane) owns 128 queries of one (utterance, head) and
// walks the keys < length in tiles of 64, twice (the skeleton of attention_train.cu's FWD mode):
//   pass A: S_j = Q K_j^T -> exact row max and sum -> log-sum-exp;
//   pass B: S_j again, P_j = 2^(s - lse) in [0, 1] (already normalised), O += P_j V_j.
// Q and K are split in shared memory as loaded (K-major: the head dimension is contiguous); V is split AND
// transposed into a K-major [d][key] tile, so every MMA operand is K-major; P is split by the thread that owns
// its row.  The raw K / V buffer is free once split, so the next tile's TMA overlaps this tile's MMAs and
// softmax.  No L x L buffer: any L the TMA box walk reaches.
constexpr int AX_HD = 64;
constexpr int AX_OWN = 128;
constexpr int AX_OTH = 64;
constexpr int AX_Q_ATOM = AX_OWN * 128;  // 16 KB: 128 rows x 32 fp32
constexpr int AX_K_ATOM = AX_OTH * 128;  //  8 KB
constexpr int AX_SMEM = 4 * AX_Q_ATOM /*Q hi, lo*/ + 4 * AX_K_ATOM /*raw K, V*/ + 4 * AX_K_ATOM /*K hi, lo*/ +
                        4 * AX_K_ATOM /*V^T hi, lo*/ + 4 * AX_Q_ATOM /*P hi, lo*/ + 64 /*barriers*/ + 1024;

struct AttnX3Params {
  float* out;           // [L*B, D]
  const int* lengths;   // [B]
  const int* q_limit;   // device [1] or NULL
  int L, B, H;
  float scale_log2e;    // the scores arrive pre-scaled (head_dim^-0.5 folded into q): log2(e)
  int log_penalty;
};

__device__ __forceinline__ float ax_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// byte offset of element (row, col) in a K-major 128-byte-swizzled atom of 32 fp32 columns
__device__ __forceinline__ int sw_off(int row, int col) {
  return row * 128 + ((((col >> 2) ^ (row & 7))) << 4) + ((col & 3) << 2);
}

__global__ void __launch_bounds__(128, 1)
    attn_tf32x3_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                       const AttnX3Params p) {
  const int L = p.L, B = p.B, H = p.H, D = H * AX_HD;
  const int bh = blockIdx.y, b = bh / H, h = bh - b * H;
  const int r0 = blockIdx.x * AX_OWN;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int row = r0 + tid;
  const int len = min(__ldg(p.lengths + b), L);
  if (p.q_limit != nullptr && r0 >= __ldg(p.q_limit)) return;  // the caller never reads these rows
  if (r0 >= len) {  // only padded queries: defined zeros (CTA-uniform)
    if (row < L) {
      float4* op = reinterpret_cast<float4*>(p.out + ((size_t)row * B + b) * D + h * AX_HD);
#pragma unroll
      for (int c = 0; c < 16; ++c) op[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    return;
  }

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sQhi = smem;                     // 2 atoms (d 0-31 | 32-63), split in place
  uint8_t* sQlo = sQhi + 2 * AX_Q_ATOM;
  uint8_t* sRaw = sQlo + 2 * AX_Q_ATOM;     // K atoms 0,1 | V atoms 0,1 (raw fp32 from TMA)
  uint8_t* sKhi = sRaw + 4 * AX_K_ATOM;
  uint8_t* sKlo = sKhi + 2 * AX_K_ATOM;
  uint8_t* sVhi = sKlo + 2 * AX_K_ATOM;     // V^T: rows d, 2 atoms over keys 0-31 | 32-63
  uint8_t* sVlo = sVhi + 2 * AX_K_ATOM;
  uint8_t* sPhi = sVlo + 2 * AX_K_ATOM;     // rows = queries, 2 atoms over keys 0-31 | 32-63
  uint8_t* sPlo = sPhi + 2 * AX_Q_ATOM;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sPlo + 2 * AX_Q_ATOM);
  uint64_t* bar_q = bars + 0;
  uint64_t* bar_ld = bars + 1;
  uint64_t* bar_s = bars + 2;
  uint64_t* bar_o = bars + 3;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);

  if (tid == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    mbar_init(bar_q, 1);
    mbar_init(bar_ld, 1);
    mbar_init(bar_s, 1);
    mbar_init(bar_o, 1);
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 0) {
    tmem_alloc(tmem_slot, 128);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t lane_addr = static_cast<uint32_t>(warp * 32) << 16;
  const uint32_t tS = tmem_base + lane_addr;       // columns  0..63: S
  const uint32_t tO = tmem_base + lane_addr + 64;  // columns 64..127: O

  constexpr uint32_t IDESC = idesc_tf32_f32(AX_OWN, 64);
  const int cq = h * AX_HD, ck = D + h * AX_HD, cv = 2 * D + h * AX_HD;
  const int n_k = (len + AX_OTH - 1) / AX_OTH;
  const int n_steps = 2 * n_k;  // pass A: steps 0 .. n_k-1 (K only); pass B: n_k .. 2 n_k - 1 (K and V)

  auto issue_load = [&](int s) {
    const int j = s < n_k ? s : s - n_k;
    const bool with_v = s >= n_k;
    mbar_arrive_expect_tx(bar_ld, (with_v ? 4 : 2) * AX_K_ATOM);
    tma_load_3d(sRaw, &tmKV, bar_ld, ck, b, j * AX_OTH);
    tma_load_3d(sRaw + AX_K_ATOM, &tmKV, bar_ld, ck + 32, b, j * AX_OTH);
    if (with_v) {
      tma_load_3d(sRaw + 2 * AX_K_ATOM, &tmKV, bar_ld, cv, b, j * AX_OTH);
      tma_load_3d(sRaw + 3 * AX_K_ATOM, &tmKV, bar_ld, cv + 32, b, j * AX_OTH);
    }
  };
  if (tid == 0) {
    mbar_arrive_expect_tx(bar_q, 2 * AX_Q_ATOM);
    tma_load_3d(sQhi, &tmQ, bar_q, cq, b, r0);
    tma_load_3d(sQhi + AX_Q_ATOM, &tmQ, bar_q, cq + 32, b, r0);
    issue_load(0);
  }
  mbar_wait(bar_q, 0);
  {
    float4* q4 = reinterpret_cast<float4*>(sQhi);
    float4* l4 = reinterpret_cast<float4*>(sQlo);
    for (int i = tid; i < 2 * AX_Q_ATOM / 16; i += 128) {
      float4 hi, lo;
      split4(q4[i], hi, lo);
      q4[i] = hi;
      l4[i] = lo;
    }
  }

  uint32_t ph_ld = 0, ph_s = 0, ph_o = 0;
  float m_run = -INFINITY, l_run = 0.0f, lse2 = 0.0f;
  for (int s = 0; s < n_steps; ++s) {
    const int j = s < n_k ? s : s - n_k;
    const bool pass_b = s >= n_k;
    if (s == n_k) lse2 = m_run + __log2f(l_run);  // key 0 is always valid: m_run finite, l_run >= 1
    mbar_wait(bar_ld, ph_ld);
    ph_ld ^= 1;
    // ---- split K (and V, transposed) out of the raw buffer; keys >= len become zeros (0 * garbage = NaN)
    {
      const float4* r4 = reinterpret_cast<const float4*>(sRaw);
      float4* h4 = reinterpret_cast<float4*>(sKhi);
      float4* l4 = reinterpret_cast<float4*>(sKlo);
#pragma unroll 2
      for (int i = tid; i < 2 * AX_K_ATOM / 16; i += 128) {
        float4 hi, lo;
        split4(r4[i], hi, lo);
        h4[i] = hi;
        l4[i] = lo;
      }
      if (pass_b) {
        const int d = tid & 63, kh = tid >> 6;  // this thread: row d of V^T, keys 32 kh .. 32 kh + 31
        const uint8_t* vsrc = sRaw + 2 * AX_K_ATOM + (d >> 5) * AX_K_ATOM;
        uint8_t* dh = sVhi + kh * AX_K_ATOM;
        uint8_t* dl = sVlo + kh * AX_K_ATOM;
#pragma unroll 2
        for (int c = 0; c < 8; ++c) {
          float4 v;
          float* vv = reinterpret_cast<float*>(&v);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int key = kh * 32 + c * 4 + e;
            const float x = *reinterpret_cast<const float*>(vsrc + sw_off(key, d & 31));
            vv[e] = (j * AX_OTH + key < len) ? x : 0.0f;
          }
          float4 hi, lo;
          split4(v, hi, lo);
          *reinterpret_cast<float4*>(dh + sw_off(d, c * 4)) = hi;
          *reinterpret_cast<float4*>(dl + sw_off(d, c * 4)) = lo;
        }
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();  // raw buffer consumed; split tiles (and, at s == 0, Q) visible to the tensor core
    if (tid == 0) {
      tc_fence_after();
      if (s + 1 < n_steps) issue_load(s + 1);
      const uint32_t qh = smem_u32(sQhi), ql = smem_u32(sQlo), kh = smem_u32(sKhi), kl = smem_u32(sKlo);
#pragma unroll 1
      for (int k = 0; k < AX_HD / 8; ++k) {
        const int atom = k >> 2, u = 2 * (k & 3);
        umma_tf32x3(tS, desc_kmajor_sw128(qh + atom * AX_Q_ATOM) + u, desc_kmajor_sw128(ql + atom * AX_Q_ATOM) + u,
                    desc_kmajor_sw128(kh + atom * AX_K_ATOM) + u, desc_kmajor_sw128(kl + atom * AX_K_ATOM) + u,
                    IDESC, k != 0);
      }
      umma_commit(bar_s);
    }
    mbar_wait(bar_s, ph_s);
    ph_s ^= 1;
    tc_fence_after();
    // 32 columns at a time (a whole 64-column row in registers spills)
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      float s2[32];
      {
        uint32_t v[32];
        tmem_ld32(tS + half * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          const int k = j * AX_OTH + half * 32 + c;
          const int dist = abs(k - row);
          const float pen = (p.log_penalty && dist > 1) ? __log2f((float)dist) : 0.0f;
          const float x = __uint_as_float(v[c]) * p.scale_log2e - pen;
          s2[c] = (k < len) ? x : -INFINITY;
        }
      }
      if (!pass_b) {
        float tm = -INFINITY;
#pragma unroll
        for (int c = 0; c < 32; ++c) tm = fmaxf(tm, s2[c]);
        const float m_new = fmaxf(m_run, tm);
        if (m_new != -INFINITY) {
          float acc = 0.0f;
#pragma unroll
          for (int c = 0; c < 32; ++c) acc += ax_ex2(s2[c] - m_new);
          l_run = l_run * ax_ex2(m_run - m_new) + acc;
          m_run = m_new;
        }
      } else {
        // P_j (normalised, in [0, 1]) split into hi / lo rows of the A operand
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          float4 pv = make_float4(ax_ex2(s2[4 * c] - lse2), ax_ex2(s2[4 * c + 1] - lse2),
                                  ax_ex2(s2[4 * c + 2] - lse2), ax_ex2(s2[4 * c + 3] - lse2));
          float4 hi, lo;
          split4(pv, hi, lo);
          *reinterpret_cast<float4*>(sPhi + half * AX_Q_ATOM + sw_off(tid, c * 4)) = hi;
          *reinterpret_cast<float4*>(sPlo + half * AX_Q_ATOM + sw_off(tid, c * 4)) = lo;
        }
      }
    }
    if (!pass_b) continue;  // the next split's __syncthreads orders these S reads before the next S MMA
    // ---- pass B: O += P_j V_j
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      const uint32_t ph = smem_u32(sPhi), pl = smem_u32(sPlo), vh = smem_u32(sVhi), vl = smem_u32(sVlo);
#pragma unroll 1
      for (int k = 0; k < AX_OTH / 8; ++k) {
        const int atom = k >> 2, u = 2 * (k & 3);
        umma_tf32x3(tO, desc_kmajor_sw128(ph + atom * AX_Q_ATOM) + u, desc_kmajor_sw128(pl + atom * AX_Q_ATOM) + u,
                    desc_kmajor_sw128(vh + atom * AX_K_ATOM) + u, desc_kmajor_sw128(vl + atom * AX_K_ATOM) + u,
                    IDESC, (j > 0) || k != 0);
      }
      umma_commit(bar_o);
    }
    // P, V^T and S are reused by the next step: wait for this step's accumulation to finish reading them
    mbar_wait(bar_o, ph_o);
    ph_o ^= 1;
    tc_fence_after();
  }

  // ---- epilogue: O -> fp32 global (one row per thread, 256 contiguous bytes; tcgen05.ld is warp-collective)
  float* op = p.out + ((size_t)row * B + b) * D + h * AX_HD;
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    uint32_t v[32];
    tmem_ld32(tO + half * 32, v);
    tmem_ld_wait();
    if (row < L) {
#pragma unroll
      for (int c = 0; c < 8; ++c)
        reinterpret_cast<float4*>(op + half * 32)[c] =
            make_float4(__uint_as_float(v[4 * c]), __uint_as_float(v[4 * c + 1]), __uint_as_float(v[4 * c + 2]),
                        __uint_as_float(v[4 * c + 3]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 128);
  }
}

// =================================================================================== conv front end
// y[b, t1, f1, c] = bn_scale[c] * relu(bias[c] + sum_{kt,kf} w[c, kt*3+kf] x[b, 2 t1 - 1 + kt, 2 f1 - 1 + kf])
//                   + bn_shift[c]      (zero padding 1, stride 2; conv_transformer.py:205-212)
__global__ void conv1_f32_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                 const float* __restrict__ bias, const float* __restrict__ scale,
                                 const float* __restrict__ shift, float* __restrict__ y, int B, int T, int F,
                                 int C, int T1, int F1) {
  const long long total = (long long)B * T1 * F1 * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    long long r = i / C;
    const int f1 = (int)(r % F1);
    r /= F1;
    const int t1 = (int)(r % T1);
    const int bb = (int)(r / T1);
    float acc = 0.0f;
#pragma unroll
    for (int kt = 0; kt < 3; ++kt) {
      const int t = 2 * t1 - 1 + kt;
      if (t < 0 || t >= T) continue;
#pragma unroll
      for (int kf = 0; kf < 3; ++kf) {
        const int f = 2 * f1 - 1 + kf;
        if (f < 0 || f >= F) continue;
        acc = fmaf(__ldg(w + c * 9 + kt * 3 + kf), __ldg(x + ((long long)bb * T + t) * F + f), acc);
      }
    }
    y[i] = fmaf(fmaxf(acc + __ldg(bias + c), 0.0f), __ldg(scale + c), __ldg(shift + c));
  }
}

// col[(b, t2, f2), (kt*3 + kf)*C + c] = y1[b, 2 t2 - 1 + kt, 2 f2 - 1 + kf, c]  (zero outside)
__global__ void conv2_im2col_f32_kernel(const float4* __restrict__ y1, float4* __restrict__ col, int B, int T1,
                                        int F1, int C, int T2, int F2) {
  const int C4 = C / 4;
  const long long total = (long long)B * T2 * F2 * 9 * C4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c4 = (int)(i % C4);
    long long r = i / C4;
    const int tap = (int)(r % 9);
    r /= 9;
    const int f2 = (int)(r % F2);
    r /= F2;
    const int t2 = (int)(r % T2);
    const int bb = (int)(r / T2);
    const int t = 2 * t2 - 1 + tap / 3, f = 2 * f2 - 1 + tap % 3;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t >= 0 && t < T1 && f >= 0 && f < F1) v = __ldg(y1 + (((long long)bb * T1 + t) * F1 + f) * C4 + c4);
    col[i] = v;
  }
}

static int grid_for(long long n, int threads) {
  long long g = (n + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 16;
  return (int)(g < cap ? (g > 0 ? g : 1) : cap);
}

}  // namespace fbkst

using namespace fbkst;

extern "C" int fbkst_linear_tf32x3(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                                   const float* col_scale, const float* col_shift, const float* residual,
                                   int64_t ldr, float* out, int64_t ldo, int M, int N, int K, int relu,
                                   const int32_t* m_limit, int m_limit_mult, fbkst_stream_t stream) {
  FBKST_REQUIRE(A && W && out, "fbkst_linear_tf32x3: null operand");
  FBKST_REQUIRE(M > 0 && N > 0 && K > 0, "fbkst_linear_tf32x3: empty problem M=%d N=%d K=%d", M, N, K);
  FBKST_REQUIRE(K % 4 == 0 && lda % 4 == 0 && ldw % 4 == 0 && lda >= K && ldw >= K,
                "fbkst_linear_tf32x3: K, lda, ldw must be multiples of 4 (K=%d lda=%lld ldw=%lld)", K,
                (long long)lda, (long long)ldw);
  FBKST_REQUIRE(ldo >= N && (residual == nullptr || ldr >= N), "fbkst_linear_tf32x3: output / residual pitch < N");
  FBKST_REQUIRE((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0,
                "fbkst_linear_tf32x3: A and W must be 16-byte aligned");
  FBKST_REQUIRE((col_scale == nullptr) == (col_shift == nullptr),
                "fbkst_linear_tf32x3: col_scale and col_shift come together");
  FBKST_REQUIRE(m_limit == nullptr || m_limit_mult > 0, "fbkst_linear_tf32x3: m_limit needs m_limit_mult > 0");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  static PerDeviceFlag configured;
  if (!configured) {
    FBKST_CHECK_CUDA(
        cudaFuncSetAttribute(gemm_tf32x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, X3_SMEM));
    configured = true;
  }
  CUtensorMap tmA, tmB;
  int rc = make_map_f32_2d(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda, X3_BM);
  if (rc) return rc;
  rc = make_map_f32_2d(&tmB, W, (uint64_t)N, (uint64_t)K, (uint64_t)ldw, X3_BN);
  if (rc) return rc;
  X3Epi ep;
  ep.bias = bias;
  ep.col_scale = col_scale;
  ep.col_shift = col_shift;
  ep.resid = residual;
  ep.ldr = ldr;
  ep.out = out;
  ep.ldo = ldo;
  ep.relu = relu;
  const int tiles = ((M + X3_BM - 1) / X3_BM) * ((N + X3_BN - 1) / X3_BN);
  const int grid = tiles < num_sms() ? tiles : num_sms();
  gemm_tf32x3_kernel<<<grid, 384, X3_SMEM, st>>>(tmA, tmB, M, N, K, m_limit, m_limit_mult, ep);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_attention_tf32x3(const float* qkv, float* out, const int32_t* lengths, int L, int B, int H,
                                      int log_penalty, const int32_t* q_limit, fbkst_stream_t stream) {
  FBKST_REQUIRE(qkv && out && lengths, "fbkst_attention_tf32x3: null pointer");
  FBKST_REQUIRE(L > 0 && B > 0 && H > 0 && H <= 16 && B * H <= 65535,
                "fbkst_attention_tf32x3: bad shape L=%d B=%d H=%d (H <= 16)", L, B, H);
  FBKST_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                "fbkst_attention_tf32x3: qkv and out must be 16-byte aligned");
  const int D = H * AX_HD;
  CUtensorMap tmQ, tmKV;
  uint64_t dims[3] = {(uint64_t)3 * D, (uint64_t)B, (uint64_t)L};
  uint64_t strides[2] = {(uint64_t)3 * D * 4, (uint64_t)B * 3 * D * 4};
  uint32_t boxq[3] = {32, 1, AX_OWN}, boxkv[3] = {32, 1, AX_OTH};
  int rc = make_tensor_map(&tmQ, qkv, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, 3, dims, strides, boxq, nullptr);
  if (rc) return rc;
  rc = make_tensor_map(&tmKV, qkv, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, 3, dims, strides, boxkv, nullptr);
  if (rc) return rc;
  AttnX3Params p;
  p.out = out;
  p.lengths = lengths;
  p.q_limit = q_limit;
  p.L = L;
  p.B = B;
  p.H = H;
  p.scale_log2e = 1.4426950408889634f;
  p.log_penalty = log_penalty;
  static PerDeviceFlag configured;
  if (!configured) {
    FBKST_CHECK_CUDA(
        cudaFuncSetAttribute(attn_tf32x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AX_SMEM));
    configured = true;
  }
  dim3 grid((L + AX_OWN - 1) / AX_OWN, B * H);
  attn_tf32x3_kernel<<<grid, 128, AX_SMEM, reinterpret_cast<cudaStream_t>(stream)>>>(tmQ, tmKV, p);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_conv1_relu_bn_f32(const float* x, const float* w, const float* bias, const float* bn_scale,
                                       const float* bn_shift, float* y, int B, int T, int F, int C,
                                       fbkst_stream_t stream) {
  FBKST_REQUIRE(x && w && bias && bn_scale && bn_shift && y, "fbkst_conv1_relu_bn_f32: null pointer");
  FBKST_REQUIRE(B > 0 && T > 0 && F > 0 && C > 0, "fbkst_conv1_relu_bn_f32: bad shape");
  const int T1 = (T + 1) / 2, F1 = (F + 1) / 2;
  const long long n = (long long)B * T1 * F1 * C;
  conv1_f32_kernel<<<grid_for(n, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x, w, bias, bn_scale, bn_shift, y, B, T, F, C, T1, F1);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_conv2_im2col_f32(const float* y1, float* col, int B, int T1, int F1, int C,
                                      fbkst_stream_t stream) {
  FBKST_REQUIRE(y1 && col, "fbkst_conv2_im2col_f32: null pointer");
  FBKST_REQUIRE(B > 0 && T1 > 0 && F1 > 0 && C > 0 && C % 4 == 0, "fbkst_conv2_im2col_f32: bad shape (C %% 4 == 0)");
  FBKST_REQUIRE((reinterpret_cast<uintptr_t>(y1) & 15) == 0 && (reinterpret_cast<uintptr_t>(col) & 15) == 0,
                "fbkst_conv2_im2col_f32: 16-byte aligned buffers required");
  const int T2 = (T1 + 1) / 2, F2 = (F1 + 1) / 2;
  const long long n = (long long)B * T2 * F2 * 9 * (C / 4);
  conv2_im2col_f32_kernel<<<grid_for(n, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(y1), reinterpret_cast<float4*>(col), B, T1, F1, C, T2, F2);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}
