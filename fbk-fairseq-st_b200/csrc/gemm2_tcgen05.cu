// out = epilogue(A @ W^T) with CTA-PAIR tensor-core tiles (tcgen05 cta_group::2).
//
// A single-CTA kernel with 128x256 tiles (since removed) moves 48 KB of operands from L2 per 128x256x64 MMA
// block, i.e. 94 B/clk/SM at full tensor rate -- more than twice what L2 can deliver to 148 SMs
// (measured: the kernel saturates at ~11.5 TB/s of L2->SM traffic, ~50% tensor-pipe utilisation).
// Here two CTAs of a cluster (one TPC) compute ONE 256x256 tile: each CTA stages its own 128 rows
// of A and HALF of the W tile (128 of the 256 columns); the leader CTA issues
// tcgen05.mma.cta_group::2 (M=256, N=256), which reads both halves of W from both CTAs' shared
// memory and writes each CTA's 128 accumulator rows into that CTA's TMEM.  Operand traffic per
// FLOP drops by 1.5x, the smem ring gets 5 stages of 32 KB, and the epilogue staging buffers are
// double-buffered.
//
// Per CTA: warp 0 TMA producer (loads signal the LEADER's full barrier), warp 1 MMA issuer
// (leader only; commits are multicast to both CTAs), warp 2 TMEM allocator, warps 4-11 epilogue
// (TMEM -> registers -> bias/ReLU/residual -> swizzled smem -> per-warp TMA store).
#include "host_common.h"
#include "ptx.cuh"

namespace fbkst {

constexpr int G2_BM = 128;      // rows per CTA (256 per pair)
constexpr int G2_BN = 256;      // tile columns (each CTA stages 128 of them)
constexpr int G2_BK = 64;
constexpr int G2_A_BYTES = G2_BM * G2_BK * 2;        // 16 KB
constexpr int G2_B_BYTES = (G2_BN / 2) * G2_BK * 2;  // 16 KB
constexpr int G2_STAGE_BYTES = G2_A_BYTES + G2_B_BYTES;
constexpr int G2_EPI_BYTES = 8 * 2 * 4096;
constexpr int G2_XB_BYTES = 8 * 4096;  // LNS: per-warp staging of the bf16 copy (32 rows x 64 columns)
// The LayerNorm-statistics variant trades one operand stage for the bf16 staging buffers.
constexpr int g2_stages(bool lns) { return lns ? 4 : 5; }
constexpr int g2_smem(bool lns) {
  return g2_stages(lns) * G2_STAGE_BYTES + G2_EPI_BYTES + (lns ? G2_XB_BYTES : 0) + 512 + 1024;
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local_addr` (a shared::cta address) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
// Remote arrive on the LEADER's "accumulator free" barrier.  RELAXED on purpose: the only thing
// the leader's MMA must not overtake is our tcgen05.ld of the accumulator, which has completed
// (tcgen05.wait::ld) and is ordered by tcgen05.fence::before_thread_sync; no ordinary memory is
// handed over.  `.release.cluster` compiled to MEMBAR.ALL.GPU + CCTL.IVALL per tile and warp --
// 46 % of the epilogue warps' stall samples (profiles/r01a_ncu_gemm2.txt).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr)
               : "memory");
}
__device__ __forceinline__ void tmem_alloc_cg2(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_cg2() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cg2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// TMA load whose completion bytes are credited to an mbarrier given as a shared::cluster address
// (the leader CTA's full barrier), as both CTAs of the pair feed one MMA.
__device__ __forceinline__ void tma_load_2d_cg2(void* smem_dst, const void* tmap, uint32_t mbar_cluster,
                                                int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
      "l"(tmap), "r"(mbar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_ss_cg2(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                                 uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (count 1) on the barrier at the same smem offset in every CTA of `cta_mask` once all
// tcgen05.mma issued so far by this thread have completed
__device__ __forceinline__ void umma_commit_cg2_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::
          "r"(smem_u32(bar)),
      "h"(cta_mask)
      : "memory");
}
__device__ __forceinline__ float4 bcast4_g2(const float4& v, int src_lane) {
  return make_float4(__shfl_sync(0xffffffffu, v.x, src_lane), __shfl_sync(0xffffffffu, v.y, src_lane),
                     __shfl_sync(0xffffffffu, v.z, src_lane), __shfl_sync(0xffffffffu, v.w, src_lane));
}

// LayerNorm folded into the GEMMs around it (the reference's pre-LN block,
// fairseq/modules/transformer_layer.py:108-133: x = x + f(LN(x))):
//   LN(x) W^T + b = rstd * (x W''^T) + c,   W''[n,k] = gamma[k] W[n,k] - mean_k(gamma[k] W[n,k]),
//                                           c[n] = b[n] + sum_k beta[k] W[n,k]
// (the row mean drops out because every row of W'' sums to zero).  So the PRODUCER of x (out_proj /
// fc2, LNS = true) also emits bf16(x) and, per row and 128-column slice, the (mean, M2) of that slice;
// the CONSUMER (QKV / fc1, ln_stats != nullptr) merges the slices (Chan), and its epilogue is
// fma(rstd, acc, c) instead of acc + b.  No LayerNorm kernel, no fp32 re-read of x.
struct LnStatsIn {
  const float2* stats;  // [M, parts] (mean, M2) per 128-column slice of the consumer's K dimension
  int parts;
  int dim;  // LayerNorm width (== K)
  float eps;
};

// (mean, M2) of `parts` slices -> 1/sqrt(var + eps); slice p covers min(128, dim - 128 p) columns
__device__ __forceinline__ float ln_rstd_from_slices(const float2* __restrict__ st, int parts, int dim,
                                                     float eps) {
  float n = 0.f, mean = 0.f, m2 = 0.f;
  for (int p = 0; p < parts; ++p) {
    const float2 v = __ldg(st + p);
    const float c = (float)min(128, dim - 128 * p);
    const float tot = n + c, delta = v.x - mean;
    mean += delta * (c / tot);
    m2 += v.y + delta * delta * (n * c / tot);
    n = tot;
  }
  return rsqrtf(m2 / (float)dim + eps);
}

// CTC projection epilogue (AM): while the fp32 logits of a tile pass through the epilogue registers, every
// thread (= one output row) also folds its <= 128 columns into (max, first arg-max, sum of exp(x - max)) and
// writes that partial to partial[row, chunk]; a tiny merge kernel (ctc.cu) turns the ceil(N/128) partials of a
// row into the frame's label / top probability / log-sum-exp.  The 4-byte-per-element re-read of the logits
// by a separate arg-max pass (768 MB at cfg2) disappears (SURVEY 8d, VERDICT r01 #6).  `bump_cols[row]`
// (optional) adds `bump` to one column per row BEFORE the store and the arg-max: the run-structured logit
// injection of the benchmarks / parity tests (SURVEY F9), equivalent to a forward hook on ctc_fc.
struct ArgmaxEpi {
  float4* partial;       // [M, chunks] (max, index as float bits, sum, -)
  const int* bump_cols;  // [M] or nullptr
  float bump;
  int want_sum;
  int chunks;
};

// MNM: both operands are MN-major ("TN" weight-gradient product dW[n, k] = sum_t g[t, n] x[t, k], operands
// in their natural token-major layouts): tmA / tmB are maps of the [tokens, n_out] / [tokens, k_in] matrices
// with {64 (MN), 64 (tokens)} boxes; a CTA's 128 MN rows are two such boxes 8 KB apart (descriptor LBO), a
// 16-token k-step advances the start address by 16 rows x 128 B.
template <bool OUT_F32, bool RESID, bool LNS, bool AM = false, bool MNM = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(384, 1)
    gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmR,
                 const __grid_constant__ CUtensorMap tmX, int M, int N, int K,
                 const float* __restrict__ bias, int relu, const int* __restrict__ m_limit,
                 int m_limit_mult, const LnStatsIn ln_in, float2* __restrict__ stats_out,
                 const uint32_t idesc, const int splits, const int split_rows, const ArgmaxEpi am) {
  static_assert(!LNS || (OUT_F32 && RESID), "row statistics are produced by the residual epilogue");
  static_assert(!AM || (OUT_F32 && !RESID), "the arg-max epilogue rides on the plain fp32 store");
  constexpr int G2_STAGES = g2_stages(LNS);
  constexpr uint32_t TMEM_COLS = 512;  // two 256-column accumulator stages

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* smem_epi = smem + G2_STAGES * G2_STAGE_BYTES;
  uint8_t* smem_xb = smem_epi + G2_EPI_BYTES;  // LNS only
  uint64_t* full_bar =
      reinterpret_cast<uint64_t*>(smem_epi + G2_EPI_BYTES + (LNS ? G2_XB_BYTES : 0));  // used in the leader
  uint64_t* empty_bar = full_bar + G2_STAGES;                                 // per CTA
  uint64_t* tfull_bar = empty_bar + G2_STAGES;                                // per CTA
  uint64_t* tempty_bar = tfull_bar + 2;                                       // used in the leader
  uint64_t* res_bar = tempty_bar + 2;                                         // [8][2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + 16);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int cluster_id = blockIdx.x >> 1;
  const int num_clusters = gridDim.x >> 1;
  pdl_launch_dependents();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmO);
    if (RESID) tma_prefetch_desc(&tmR);
    if (LNS) tma_prefetch_desc(&tmX);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < G2_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], 16);  // 8 epilogue warps x 2 CTAs
    }
    for (int s = 0; s < 16; ++s) mbar_init(&res_bar[s], 1);
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc_cg2(tmem_slot, TMEM_COLS);
    tmem_relinquish_cg2();
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Everything above is independent of the previous kernel's output (PDL prologue); nothing below
  // may run before that kernel has completed.
  pdl_wait();
  // device-side row limit (rows valid after CTC compression): tiles beyond it are skipped
  if (m_limit != nullptr) M = min(M, __ldg(m_limit) * m_limit_mult);
  const int num_n = (N + G2_BN - 1) / G2_BN;
  const int num_m = (M + 2 * G2_BM - 1) / (2 * G2_BM);
  const int num_kb = (K + G2_BK - 1) / G2_BK;
  // Split-K (wgrad: few output tiles, K = tokens): tile index = (split, m_blk, n_blk); split s covers
  // k-blocks [s*kb_per, min(num_kb, (s+1)*kb_per)) and stores its partial product at output rows
  // m + s*split_rows (a [splits, split_rows, N] buffer reduced by a second kernel).  splits == 1: the
  // ordinary GEMM.  The host guarantees that no split is empty.
  const int tiles_mn = num_m * num_n;
  const int num_tiles = tiles_mn * splits;
  const int kb_per = (num_kb + splits - 1) / splits;

  // Producer and MMA warps run in warp-uniform control flow and let ONE ELECTED lane issue: under
  // `if (lane == 0)` ptxas wraps every UTMALDG / UTCHMMA in a divergence waterfall (ELECT +
  // BRA.U.ANY loop, descriptors rebuilt per instruction); uniform code keeps them in uniform
  // registers and issues the four MMAs of a k-block back to back.
  if (warp == 0) {
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
      const int sp = tile / tiles_mn, t2 = tile - sp * tiles_mn;
      const int m_blk = t2 / num_n, n_blk = t2 - m_blk * num_n;
      const int row_a = m_blk * 2 * G2_BM + (int)rank * G2_BM;
      const int row_b = n_blk * G2_BN + (int)rank * (G2_BN / 2);
      const int kb0 = sp * kb_per, kb1 = min(num_kb, kb0 + kb_per);
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (elect_one()) {
          if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * G2_STAGE_BYTES);
          const uint32_t leader_full = map_to_cta(smem_u32(&full_bar[stage]), 0);
          uint8_t* sa = smem + stage * G2_STAGE_BYTES;
          if (MNM) {
            tma_load_2d_cg2(sa, &tmA, leader_full, row_a, kb * G2_BK);
            tma_load_2d_cg2(sa + G2_A_BYTES / 2, &tmA, leader_full, row_a + 64, kb * G2_BK);
            tma_load_2d_cg2(sa + G2_A_BYTES, &tmB, leader_full, row_b, kb * G2_BK);
            tma_load_2d_cg2(sa + G2_A_BYTES + G2_B_BYTES / 2, &tmB, leader_full, row_b + 64, kb * G2_BK);
          } else {
            tma_load_2d_cg2(sa, &tmA, leader_full, kb * G2_BK, row_a);
            tma_load_2d_cg2(sa + G2_A_BYTES, &tmB, leader_full, kb * G2_BK, row_b);
          }
        }
        __syncwarp();
        if (++stage == G2_STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * G2_BN;
        const int sp = tile / tiles_mn;
        const int kb0 = sp * kb_per, kb1 = min(num_kb, kb0 + kb_per);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * G2_STAGE_BYTES);
          const uint64_t adesc = MNM ? desc_mnmajor_sw128(sa, G2_A_BYTES / 2) : desc_kmajor_sw128(sa);
          const uint64_t bdesc =
              MNM ? desc_mnmajor_sw128(sa + G2_A_BYTES, G2_B_BYTES / 2) : desc_kmajor_sw128(sa + G2_A_BYTES);
          constexpr int KSTEP = MNM ? (16 * 128) >> 4 : 2;  // descriptor units (16 B) per 16-element k-step
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < G2_BK / 16; ++k)
              umma_bf16_ss_cg2(d_tmem, adesc + KSTEP * k, bdesc + KSTEP * k, idesc, ((kb - kb0) | k) != 0);
            umma_commit_cg2_mc(&empty_bar[stage], 0x3);
            if (kb == kb1 - 1) umma_commit_cg2_mc(&tfull_bar[acc], 0x3);
          }
          __syncwarp();
          if (++stage == G2_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else if (warp >= 4) {
    const int ew = warp - 4;
    const int q = ew & 3;      // TMEM lane quarter == row block of 32
    const int half = ew >> 2;  // column half of the tile
    uint8_t* stg = smem_epi + ew * 2 * 4096;
    uint64_t* rbar = res_bar + ew * 2;
    uint32_t rphase[2] = {0, 0};
    int acc = 0;
    uint32_t acc_phase = 0;
    const int swz = lane & 7;
    int sbuf = 0;  // staging buffer toggle (non-residual path)
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
      const int sp = tile / tiles_mn, t2 = tile - sp * tiles_mn;
      const int m_blk = t2 / num_n, n_blk = t2 - m_blk * num_n;
      const int m_store = sp * split_rows;  // row offset of this split's partial product
      const int m0 = m_blk * 2 * G2_BM + (int)rank * G2_BM + q * 32;
      const int n0 = n_blk * G2_BN + half * 128;
      const uint32_t tempty_leader = map_to_cta(smem_u32(&tempty_bar[acc]), 0);
      if (n0 >= N || m0 >= M) {  // nothing to write for this warp (warp-uniform)
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_before();
        if (lane == 0) mbar_arrive_cluster(tempty_leader);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
        continue;
      }
      float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (bias != nullptr) {
        const int c = n0 + lane * 4;
        if (c + 3 < N) {
          b4 = __ldg(reinterpret_cast<const float4*>(bias + c));
        } else {
          if (c + 0 < N) b4.x = __ldg(bias + c + 0);
          if (c + 1 < N) b4.y = __ldg(bias + c + 1);
          if (c + 2 < N) b4.z = __ldg(bias + c + 2);
        }
      }
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * G2_BN + half * 128;
      if (RESID) {  // fp32 out, 4 units of 32 columns, residual prefetched one unit ahead
        if (lane == 0) {
          tma_store_wait_read<0>();
          mbar_arrive_expect_tx(&rbar[0], 4096);
          tma_load_2d(stg, &tmR, &rbar[0], n0, m0);
        }
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
        uint32_t v[32];
        tmem_ld32(taddr, v);
        // LNS: statistics of this thread's row over the warp's <= 128 columns, shifted by the first
        // value (single pass without cancellation), and the bf16 copy of x staged 64 columns at a time
        float ln_shift = 0.f, ln_s1 = 0.f, ln_s2 = 0.f;
        uint8_t* xrow = smem_xb + ew * 4096 + lane * 128;
#pragma unroll 1
        for (int u = 0; u < 4; ++u) {
          const int col0 = n0 + u * 32;
          if (col0 >= N) break;
          const int bsel = u & 1;
          if (u + 1 < 4 && col0 + 32 < N && lane == 0) {  // prefetch the next residual unit
            tma_store_wait_read<0>();                    // its buffer was read by store(u-1)
            mbar_arrive_expect_tx(&rbar[bsel ^ 1], 4096);
            tma_load_2d(stg + (bsel ^ 1) * 4096, &tmR, &rbar[bsel ^ 1], col0 + 32, m0);
          }
          if (LNS && bsel == 0) {  // the bf16 staging buffer was read by the store issued at unit u-1
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
          }
          tmem_ld_wait();
          float f[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
          if (u + 1 < 4) tmem_ld32(taddr + (u + 1) * 32, v);
          mbar_wait(&rbar[bsel], rphase[bsel]);
          rphase[bsel] ^= 1;
          uint8_t* rowp = stg + bsel * 4096 + lane * 128;
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const float4 bb = bcast4_g2(b4, u * 8 + g);
            float4* sp = reinterpret_cast<float4*>(rowp + ((g ^ swz) << 4));
            float4 r = *sp;
            float a0 = f[4 * g] + bb.x, a1 = f[4 * g + 1] + bb.y, a2 = f[4 * g + 2] + bb.z,
                  a3 = f[4 * g + 3] + bb.w;
            if (relu) {
              a0 = fmaxf(a0, 0.f);
              a1 = fmaxf(a1, 0.f);
              a2 = fmaxf(a2, 0.f);
              a3 = fmaxf(a3, 0.f);
            }
            r.x += a0;
            r.y += a1;
            r.z += a2;
            r.w += a3;
            *sp = r;
            if (LNS) {
              if (u == 0 && g == 0) ln_shift = r.x;
              const float d0 = r.x - ln_shift, d1 = r.y - ln_shift, d2 = r.z - ln_shift,
                          d3 = r.w - ln_shift;
              ln_s1 += (d0 + d1) + (d2 + d3);
              ln_s2 = fmaf(d0, d0, fmaf(d1, d1, fmaf(d2, d2, fmaf(d3, d3, ln_s2))));
              // columns (u&1)*32 + 4g .. +3 of the 64-column staging row: 8 bytes at offset
              // (u&1)*64 + 8g, i.e. 16-byte chunk (u&1)*4 + g/2 (XOR-swizzled), half g&1
              *reinterpret_cast<uint2*>(xrow + ((((bsel << 2) | (g >> 1)) ^ swz) << 4) + ((g & 1) << 3)) =
                  make_uint2(pack_bf16x2(r.x, r.y), pack_bf16x2(r.z, r.w));
            }
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tmO, stg + bsel * 4096, col0, m0);
            if (LNS && (bsel == 1 || col0 + 32 >= N))
              tma_store_2d(&tmX, smem_xb + ew * 4096, n0 + (u >> 1) * 64, m0);
            tma_store_commit();
          }
        }
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tempty_leader);
        if (LNS && m0 + lane < M) {
          const float cnt = (float)min(128, N - n0);
          stats_out[(size_t)(m0 + lane) * ((N + 127) >> 7) + (n0 >> 7)] =
              make_float2(ln_shift + ln_s1 / cnt, fmaxf(ln_s2 - ln_s1 * ln_s1 / cnt, 0.f));
        }
      } else {
        // folded LayerNorm: per-row 1/sigma from the producer's slice statistics (loaded before the
        // accumulator wait so the latency hides under the main loop); 1 when there is no LayerNorm
        float rs = 1.0f;
        if (ln_in.stats != nullptr && m0 + lane < M)
          rs = ln_rstd_from_slices(ln_in.stats + (size_t)(m0 + lane) * ln_in.parts, ln_in.parts,
                                   ln_in.dim, ln_in.eps);
        mbar_wait(&tfull_bar[acc], acc_phase);
        tc_fence_after();
        constexpr int UNITS = OUT_F32 ? 4 : 2;  // staging rows are 128 B: 32 fp32 or 64 bf16 columns
        constexpr int UCOLS = OUT_F32 ? 32 : 64;
        float am_best = -INFINITY, am_sum = 0.f, am_bump_val = 0.f;
        int am_idx = 0x7fffffff;
        const int am_bump = (AM && am.bump_cols != nullptr && m0 + lane < M) ? __ldg(am.bump_cols + m0 + lane) : -1;
        const bool am_tail = AM && (n0 + 128 > N);
#pragma unroll 1
        for (int u = 0; u < UNITS; ++u) {
          const int col0 = n0 + u * UCOLS;
          if (col0 >= N) break;
          uint32_t v0[32], v1[32];
          tmem_ld32(taddr + u * UCOLS, v0);
          if (!OUT_F32) tmem_ld32(taddr + u * UCOLS + 32, v1);
          if (lane == 0) tma_store_wait_read<1>();  // the buffer used two units ago is free again
          tmem_ld_wait();
          if (u == UNITS - 1 || col0 + UCOLS >= N) {  // all TMEM reads of this tile done: release it
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(tempty_leader);
          }
          __syncwarp();
          uint8_t* rowp = stg + sbuf * 4096 + lane * 128;
          if (OUT_F32) {
#pragma unroll
            for (int g = 0; g < 8; ++g) {
              const float4 bb = bcast4_g2(b4, u * 8 + g);
              float a0 = fmaf(rs, __uint_as_float(v0[4 * g]), bb.x),
                    a1 = fmaf(rs, __uint_as_float(v0[4 * g + 1]), bb.y),
                    a2 = fmaf(rs, __uint_as_float(v0[4 * g + 2]), bb.z),
                    a3 = fmaf(rs, __uint_as_float(v0[4 * g + 3]), bb.w);
              if (relu) {
                a0 = fmaxf(a0, 0.f);
                a1 = fmaxf(a1, 0.f);
                a2 = fmaxf(a2, 0.f);
                a3 = fmaxf(a3, 0.f);
              }
              if (AM && !am.want_sum) {
                // LEAN form (no sum exp wanted): only the row maximum of the chunk, two FMNMX3 per four logits.
                // The arg-max column is recovered by the merge kernel from the ONE winning chunk of the row
                // (128 logits re-read per row: 12 MB of the 771 MB at cfg2); the bumped logit is folded in
                // after the loop from the staging row.
                const int c = col0 + 4 * g;
                float x0 = a0, x1 = a1, x2 = a2, x3 = a3;
                if (am_tail) {  // tile-uniform: only the last column tile
                  x0 = (c < N) ? a0 : -INFINITY;
                  x1 = (c + 1 < N) ? a1 : -INFINITY;
                  x2 = (c + 2 < N) ? a2 : -INFINITY;
                  x3 = (c + 3 < N) ? a3 : -INFINITY;
                }
                am_best = fmaxf(fmaxf(am_best, x0), fmaxf(fmaxf(x1, x2), x3));
              } else if (AM) {
                // running (max, first arg-max, sum exp) of this row over the warp's columns.  ~1.5 instructions
                // per element: the max changes O(log n) times per row, so the update branch is rare.  The logit
                // bump and the columns >= N of the last tile are handled outside this loop.
                const int c = col0 + 4 * g;
                float x0 = a0, x1 = a1, x2 = a2, x3 = a3;
                if (am_tail) {  // tile-uniform: only the last column tile
                  x0 = (c < N) ? a0 : -INFINITY;
                  x1 = (c + 1 < N) ? a1 : -INFINITY;
                  x2 = (c + 2 < N) ? a2 : -INFINITY;
                  x3 = (c + 3 < N) ? a3 : -INFINITY;
                }
                const float m4 = fmaxf(fmaxf(x0, x1), fmaxf(x2, x3));
                if (m4 > am_best) {  // strict: an earlier (lower) column keeps equal values
                  if (am.want_sum) am_sum *= exp2f((am_best - m4) * 1.4426950408889634f);
                  am_best = m4;
                  am_idx = c + ((x0 == m4) ? 0 : (x1 == m4) ? 1 : (x2 == m4) ? 2 : 3);
                }
                if (am.want_sum) {
                  const float nb = -am_best * 1.4426950408889634f;
                  am_sum += (exp2f(fmaf(x0, 1.4426950408889634f, nb)) + exp2f(fmaf(x1, 1.4426950408889634f, nb))) +
                            (exp2f(fmaf(x2, 1.4426950408889634f, nb)) + exp2f(fmaf(x3, 1.4426950408889634f, nb)));
                }
                if (am_bump >= c && am_bump < c + 4)  // remember the un-bumped logit of the bump column
                  am_bump_val = (am_bump == c) ? a0 : (am_bump == c + 1) ? a1 : (am_bump == c + 2) ? a2 : a3;
              }
              *reinterpret_cast<float4*>(rowp + ((g ^ swz) << 4)) = make_float4(a0, a1, a2, a3);
            }
          } else {
#pragma unroll
            for (int g = 0; g < 8; ++g) {
              const uint32_t* src = (g < 4) ? v0 : v1;
              const int o = (g & 3) * 8;
              const float4 b0 = bcast4_g2(b4, u * 16 + 2 * g);
              const float4 b1 = bcast4_g2(b4, u * 16 + 2 * g + 1);
              float a[8] = {fmaf(rs, __uint_as_float(src[o]), b0.x),     fmaf(rs, __uint_as_float(src[o + 1]), b0.y),
                            fmaf(rs, __uint_as_float(src[o + 2]), b0.z), fmaf(rs, __uint_as_float(src[o + 3]), b0.w),
                            fmaf(rs, __uint_as_float(src[o + 4]), b1.x), fmaf(rs, __uint_as_float(src[o + 5]), b1.y),
                            fmaf(rs, __uint_as_float(src[o + 6]), b1.z), fmaf(rs, __uint_as_float(src[o + 7]), b1.w)};
              if (relu) {
#pragma unroll
                for (int j = 0; j < 8; ++j) a[j] = fmaxf(a[j], 0.f);
              }
              *reinterpret_cast<uint4*>(rowp + ((g ^ swz) << 4)) =
                  make_uint4(pack_bf16x2(a[0], a[1]), pack_bf16x2(a[2], a[3]), pack_bf16x2(a[4], a[5]),
                             pack_bf16x2(a[6], a[7]));
            }
          }
          if (AM && am_bump >= col0 && am_bump < col0 + UCOLS) {  // the stored logit carries the bump as well
            const int j = am_bump - col0;
            float* e = reinterpret_cast<float*>(rowp + (((j >> 2) ^ swz) << 4)) + (j & 3);
            if (!am.want_sum) am_bump_val = *e;  // (lean form: the un-bumped logit was not tracked in the loop)
            *e += am.bump;
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tmO, stg + sbuf * 4096, col0, m0 + m_store);
            tma_store_commit();
          }
          sbuf ^= 1;
        }
        if (AM && m0 + lane < M) {
          if (am_bump >= n0 && am_bump < n0 + 128 && am_bump < N) {
            // fold the bumped logit in: value v = orig + bump at column am_bump (orig is already counted)
            const float v = am_bump_val + am.bump;
            if (am.want_sum) {
              const float mx = fmaxf(am_best, v);
              am_sum = am_sum * exp2f((am_best - mx) * 1.4426950408889634f) -
                       exp2f((am_bump_val - mx) * 1.4426950408889634f) + exp2f((v - mx) * 1.4426950408889634f);
            }
            if (v > am_best || (am.want_sum && v == am_best && am_bump < am_idx)) {
              am_best = v;
              am_idx = am_bump;
            }
          }
          // lean form: .y = first column of the chunk (ties between chunks resolve to the lowest), .w = 1 asks the
          // merge kernel to recover the column inside the winning chunk from the stored logits
          am.partial[(size_t)(m0 + lane) * am.chunks + (n0 >> 7)] =
              am.want_sum ? make_float4(am_best, __int_as_float(am_idx), am_sum, 0.f)
                          : make_float4(am_best, __int_as_float(n0), 0.f, 1.f);
        }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (lane == 0) tma_store_wait<0>();
  }
  tc_fence_before();
  cluster_sync_all();  // the peer's smem / TMEM must stay alive until every multicast landed
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_cg2(tmem_base, TMEM_COLS);
  }
}

template <bool OUT_F32, bool RESID, bool LNS, bool AM = false, bool MNM = false>
static int launch_gemm2(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                        const float* resid, int64_t ldr, void* out, int64_t ldo, int M, int N, int K,
                        int relu, const int* m_limit, int m_limit_mult, const LnStatsIn& ln_in,
                        void* out_bf16, int64_t ldob, float* stats_out, int ab_f16, int splits,
                        int split_rows, cudaStream_t stream, const ArgmaxEpi* am_in = nullptr) {
  constexpr int SMEM = g2_smem(LNS);
  static_assert(SMEM <= 232448, "shared memory budget exceeded");
  auto kern = gemm2_kernel<OUT_F32, RESID, LNS, AM, MNM>;
  ArgmaxEpi am{};
  if (am_in != nullptr) am = *am_in;
  static PerDeviceFlag configured;
  if (!configured) {
    FBKST_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    configured = true;
  }
  CUtensorMap tmA, tmB, tmO, tmR, tmX;
  // MNM: A is [K, M] (tokens x n_out), W is [K, N] (tokens x k_in); boxes of 64 tokens x 64 MN columns
  int rc = MNM ? make_tensor_map_2d_bf16(&tmA, A, (uint64_t)K, (uint64_t)M, (uint64_t)lda, 64, 64)
               : make_tensor_map_2d_bf16(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda, G2_BM, G2_BK);
  if (rc) return rc;
  rc = MNM ? make_tensor_map_2d_bf16(&tmB, W, (uint64_t)K, (uint64_t)N, (uint64_t)ldw, 64, 64)
           : make_tensor_map_2d_bf16(&tmB, W, (uint64_t)N, (uint64_t)K, (uint64_t)ldw, G2_BN / 2, G2_BK);
  if (rc) return rc;
  {
    uint64_t dims[2] = {(uint64_t)N, splits > 1 ? (uint64_t)splits * split_rows : (uint64_t)M};
    uint64_t strides[1] = {(uint64_t)ldo * (OUT_F32 ? 4 : 2)};
    uint32_t box[2] = {OUT_F32 ? 32u : 64u, 32u};
    rc = make_tensor_map(&tmO, out,
                         OUT_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
                         OUT_F32 ? 4 : 2, 2, dims, strides, box, nullptr);
    if (rc) return rc;
  }
  if (RESID) {
    uint64_t dims[2] = {(uint64_t)N, (uint64_t)M};
    uint64_t strides[1] = {(uint64_t)ldr * 4};
    uint32_t box[2] = {32u, 32u};
    rc = make_tensor_map(&tmR, resid, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, 2, dims, strides, box, nullptr);
    if (rc) return rc;
  } else {
    tmR = tmO;
  }
  if (LNS) {
    rc = make_tensor_map_2d_bf16(&tmX, out_bf16, (uint64_t)M, (uint64_t)N, (uint64_t)ldob, 32, 64);
    if (rc) return rc;
  } else {
    tmX = tmO;
  }
  const int tiles = ((M + 2 * G2_BM - 1) / (2 * G2_BM)) * ((N + G2_BN - 1) / G2_BN) * splits;
  const int max_clusters = num_sms() / 2;
  const int clusters = tiles < max_clusters ? tiles : max_clusters;
  FBKST_CHECK_CUDA(launch_pdl(kern, dim3(2 * clusters), dim3(384), SMEM, stream, tmA, tmB, tmO, tmR, tmX,
                              M, N, K, bias, relu, m_limit, m_limit_mult, ln_in,
                              reinterpret_cast<float2*>(stats_out),
                              MNM ? idesc_bf16_f32(256, G2_BN, 1, 1)
                                  : (ab_f16 ? idesc_f16_f32(256, G2_BN, 0, 0) : idesc_bf16_f32(256, G2_BN, 0, 0)),
                              splits, split_rows, am));
  return FBKST_OK;
}

// Entry used by fbkst_linear_bf16 / fbkst_linear_ln_bf16 (below) for the plain / residual
// epilogues.  stats_in (with its LayerNorm width == K and eps): consumer side of the folded
// LayerNorm; out_bf16 + stats_out: producer side (residual epilogue only).
int linear_pair_dispatch(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                         const float* resid, int64_t ldr, void* out, int64_t ldo, int M, int N, int K,
                         int relu, int out_f32, const int* m_limit, int m_limit_mult,
                         const float* stats_in, float ln_eps, void* out_bf16, int64_t ldob,
                         float* stats_out, int ab_f16, cudaStream_t stream) {
  LnStatsIn ln_in;
  ln_in.stats = reinterpret_cast<const float2*>(stats_in);
  ln_in.parts = (K + 127) / 128;
  ln_in.dim = K;
  ln_in.eps = ln_eps;
  if (stats_out != nullptr)
    return launch_gemm2<true, true, true>(A, lda, W, ldw, bias, resid, ldr, out, ldo, M, N, K, relu,
                                          m_limit, m_limit_mult, ln_in, out_bf16, ldob, stats_out, ab_f16, 1, 0, stream);
  if (resid != nullptr)
    return launch_gemm2<true, true, false>(A, lda, W, ldw, bias, resid, ldr, out, ldo, M, N, K, relu,
                                           m_limit, m_limit_mult, ln_in, nullptr, 0, nullptr, ab_f16, 1, 0, stream);
  if (out_f32)
    return launch_gemm2<true, false, false>(A, lda, W, ldw, bias, nullptr, 0, out, ldo, M, N, K, relu,
                                            m_limit, m_limit_mult, ln_in, nullptr, 0, nullptr, ab_f16, 1, 0, stream);
  return launch_gemm2<false, false, false>(A, lda, W, ldw, bias, nullptr, 0, out, ldo, M, N, K, relu,
                                           m_limit, m_limit_mult, ln_in, nullptr, 0, nullptr, ab_f16, 1, 0, stream);
}

// fp32 logits + per-row arg-max partials (see ArgmaxEpi): the ctc_fc projection of the inference path
int linear_pair_argmax(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, float* out,
                       int64_t ldo, int M, int N, int K, const int* bump_cols, float bump, int want_sum,
                       float* partial, const int* m_limit, int m_limit_mult, cudaStream_t stream) {
  LnStatsIn ln_in;
  ln_in.stats = nullptr;
  ln_in.parts = 0;
  ln_in.dim = K;
  ln_in.eps = 0.f;
  ArgmaxEpi am;
  am.partial = reinterpret_cast<float4*>(partial);
  am.bump_cols = bump_cols;
  am.bump = bump;
  am.want_sum = want_sum;
  am.chunks = (N + 127) / 128;
  return launch_gemm2<true, false, false, true>(A, lda, W, ldw, bias, nullptr, 0, out, ldo, M, N, K, 0, m_limit,
                                                m_limit_mult, ln_in, nullptr, 0, nullptr, 0, 1, 0, stream, &am);
}

// Split-K GEMM for weight gradients: partial[s, m, n] = sum over the s-th slice of K of A[m, k] W[n, k]
// (fp32, no bias), s < splits, stored at partial + (s * split_rows + m) * ldo.  split_rows >= M rounded
// up to the 32-row store granularity (the caller allocates [splits, split_rows, ldo] floats).
// *splits is clamped so that no slice is empty; the caller reduces the slices (fbkst_reduce_splits).
int linear_pair_splitk(const void* A, int64_t lda, const void* W, int64_t ldw, float* partial, int64_t ldo,
                       int M, int N, int K, int* splits, int split_rows, cudaStream_t stream) {
  const int num_kb = (K + G2_BK - 1) / G2_BK;
  int sp = *splits < 1 ? 1 : *splits;
  if (sp > num_kb) sp = num_kb;
  const int kb_per = (num_kb + sp - 1) / sp;
  sp = (num_kb + kb_per - 1) / kb_per;  // no empty slice
  *splits = sp;
  LnStatsIn ln_in;
  ln_in.stats = nullptr;
  ln_in.parts = 0;
  ln_in.dim = K;
  ln_in.eps = 0.f;
  return launch_gemm2<true, false, false>(A, lda, W, ldw, nullptr, nullptr, 0, partial, ldo, M, N, K, 0, nullptr,
                                          0, ln_in, nullptr, 0, nullptr, 0, sp, split_rows, stream);
}

// The same with both operands in their natural token-major layout (no transposed copies): partial[s, n, k] =
// sum over the s-th slice of tokens of g[t, n] x[t, k].  g [tokens, n_out] bf16, x [tokens, k_in] bf16 / fp16.
int linear_pair_splitk_nt(const void* g, int64_t ldg, const void* x, int64_t ldx, int x_f16, float* partial,
                          int64_t ldo, int n_out, int k_in, int tokens, int* splits, int split_rows,
                          cudaStream_t stream) {
  const int num_kb = (tokens + G2_BK - 1) / G2_BK;
  int sp = *splits < 1 ? 1 : *splits;
  if (sp > num_kb) sp = num_kb;
  const int kb_per = (num_kb + sp - 1) / sp;
  sp = (num_kb + kb_per - 1) / kb_per;  // no empty slice
  *splits = sp;
  LnStatsIn ln_in;
  ln_in.stats = nullptr;
  ln_in.parts = 0;
  ln_in.dim = tokens;
  ln_in.eps = 0.f;
  return launch_gemm2<true, false, false, false, true>(g, ldg, x, ldx, nullptr, nullptr, 0, partial, ldo, n_out, k_in,
                                                       tokens, 0, nullptr, 0, ln_in, nullptr, 0, nullptr, x_f16, sp,
                                                       split_rows, stream);
}

// splits for a wgrad GEMM with `tiles_mn` output tiles over K = tokens: fill the CTA pairs about twice,
// keep >= 8 k-blocks (512 tokens) per slice
static int wgrad_splits(int M, int N, int K) {
  const int tiles_mn = ((M + 2 * G2_BM - 1) / (2 * G2_BM)) * ((N + G2_BN - 1) / G2_BN);
  const int pairs = num_sms() / 2;
  int sp = (2 * pairs + tiles_mn - 1) / tiles_mn;
  const int num_kb = (K + G2_BK - 1) / G2_BK;
  const int max_sp = num_kb / 8 > 0 ? num_kb / 8 : 1;
  if (sp > max_sp) sp = max_sp;
  if (sp < 1) sp = 1;
  const int kb_per = (num_kb + sp - 1) / sp;
  return (num_kb + kb_per - 1) / kb_per;
}

}  // namespace fbkst

extern "C" int fbkst_linear_bf16(const void* A, int64_t lda, const void* W, int64_t ldw,
                                 const float* bias, const float* residual, int64_t ldr, void* out,
                                 int64_t ldo, int M, int N, int K, int flags, const int32_t* m_limit,
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
  const int relu = (flags & FBKST_EPI_RELU) ? 1 : 0;
  if (residual != nullptr)
    FBKST_REQUIRE(flags & FBKST_EPI_OUT_F32, "fbkst_linear_bf16: a residual requires fp32 output");
  return linear_pair_dispatch(A, lda, W, ldw, bias, residual, ldr, out, ldo, M, N, K, relu,
                              (flags & FBKST_EPI_OUT_F32) ? 1 : 0, m_limit, m_limit_mult, nullptr, 0.f, nullptr, 0,
                              nullptr, (flags & FBKST_EPI_AB_F16) ? 1 : 0, reinterpret_cast<cudaStream_t>(stream));
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

extern "C" long long fbkst_linear_wgrad_workspace(int n_out, int k_in, int tokens) {
  using namespace fbkst;
  const int sp = wgrad_splits(n_out, k_in, tokens);
  const long long split_rows = ((long long)n_out + 31) / 32 * 32;
  const long long ldo = ((long long)k_in + 7) / 8 * 8;
  return (long long)sp * split_rows * ldo;
}

// dW[n, k] = sum_m gT[n, m] * xT[k, m]  (fp32 out; both operands token-contiguous bf16): split-K over the
// tokens on the CTA-pair tcgen05 kernel + a fixed-order reduction of the slices.  replaces the autograd of
// every F.linear on the path (weight gradient).  workspace: fbkst_linear_wgrad_workspace(...) floats.
extern "C" int fbkst_linear_wgrad_bf16(const void* gT, int64_t ldg, const void* xT, int64_t ldx, float* workspace,
                                       float* dW, int64_t lddw, int n_out, int k_in, int tokens,
                                       fbkst_stream_t stream) {
  using namespace fbkst;
  FBKST_REQUIRE(gT && xT && workspace && dW, "fbkst_linear_wgrad_bf16: null pointer");
  FBKST_REQUIRE(n_out > 0 && k_in > 0 && tokens > 0, "fbkst_linear_wgrad_bf16: empty problem");
  FBKST_REQUIRE(ldg % 8 == 0 && ldx % 8 == 0 && ldg >= tokens && ldx >= tokens,
                "fbkst_linear_wgrad_bf16: operand pitches must be multiples of 8 and >= tokens");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int sp = wgrad_splits(n_out, k_in, tokens);
  const int split_rows = (n_out + 31) / 32 * 32;
  const int64_t ldo = ((int64_t)k_in + 7) / 8 * 8;
  int rc = linear_pair_splitk(gT, ldg, xT, ldx, workspace, ldo, n_out, k_in, tokens, &sp, split_rows, st);
  if (rc) return rc;
  return fbkst_reduce_sum(workspace, sp, (int64_t)split_rows * ldo, n_out, k_in, ldo, dW, lddw, 1.0f, stream);
}

extern "C" int fbkst_linear_wgrad_nt(const void* g, int64_t ldg, const void* x, int64_t ldx, int x_is_f16,
                                     float* workspace, float* dW, int64_t lddw, int n_out, int k_in, int tokens,
                                     fbkst_stream_t stream) {
  using namespace fbkst;
  FBKST_REQUIRE(g && x && workspace && dW, "fbkst_linear_wgrad_nt: null pointer");
  FBKST_REQUIRE(n_out > 0 && k_in > 0 && tokens > 0, "fbkst_linear_wgrad_nt: empty problem");
  // (one tcgen05.mma takes both operands in the SAME 16-bit format: a bf16 x fp16 product is an illegal instruction)
  FBKST_REQUIRE(!x_is_f16, "fbkst_linear_wgrad_nt: fp16 activations are not supported (use fbkst_linear_wgrad_bf16)");
  FBKST_REQUIRE(ldg % 8 == 0 && ldx % 8 == 0 && ldg >= n_out && ldx >= k_in,
                "fbkst_linear_wgrad_nt: operand pitches must be multiples of 8 and >= the row length");
  FBKST_REQUIRE((reinterpret_cast<uintptr_t>(g) & 15) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0,
                "fbkst_linear_wgrad_nt: operands must be 16-byte aligned");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int sp = wgrad_splits(n_out, k_in, tokens);
  const int split_rows = (n_out + 31) / 32 * 32;
  const int64_t ldo = ((int64_t)k_in + 7) / 8 * 8;
  int rc = linear_pair_splitk_nt(g, ldg, x, ldx, x_is_f16, workspace, ldo, n_out, k_in, tokens, &sp, split_rows, st);
  if (rc) return rc;
  return fbkst_reduce_sum(workspace, sp, (int64_t)split_rows * ldo, n_out, k_in, ldo, dW, lddw, 1.0f, stream);
}

extern "C" int fbkst_linear_wgrad_slices_bf16(const void* gT, int64_t ldg, const void* xT, int64_t ldx,
                                              float* workspace, int n_out, int k_in, int tokens, int* splits,
                                              fbkst_stream_t stream) {
  using namespace fbkst;
  FBKST_REQUIRE(gT && xT && workspace && splits, "fbkst_linear_wgrad_slices_bf16: null pointer");
  FBKST_REQUIRE(n_out > 0 && k_in > 0 && tokens > 0, "fbkst_linear_wgrad_slices_bf16: empty problem");
  FBKST_REQUIRE(ldg % 8 == 0 && ldx % 8 == 0 && ldg >= tokens && ldx >= tokens,
                "fbkst_linear_wgrad_slices_bf16: operand pitches must be multiples of 8 and >= tokens");
  int sp = wgrad_splits(n_out, k_in, tokens);
  const int split_rows = (n_out + 31) / 32 * 32;
  const int64_t ldo = ((int64_t)k_in + 7) / 8 * 8;
  int rc = linear_pair_splitk(gT, ldg, xT, ldx, workspace, ldo, n_out, k_in, tokens, &sp, split_rows,
                              reinterpret_cast<cudaStream_t>(stream));
  *splits = sp;
  return rc;
}

/* a9 + a10 step 1 fused: logits = A W^T + bias (fp32, pitch ldo) AND, per row, the arg-max partials of every
 * 128-column chunk (partial: [M, ceil(N/128)] float4), optionally after adding `bump` to column bump_cols[row].
 * Follow with fbkst_ctc_argmax_merge.  replaces conv_transformer.py:279 + :282-284 without re-reading the logits. */
extern "C" int fbkst_linear_argmax_f32(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                                       float* out, int64_t ldo, int M, int N, int K, const int32_t* bump_cols,
                                       float bump, int want_sum, float* partial, const int32_t* m_limit,
                                       int m_limit_mult, fbkst_stream_t stream) {
  using namespace fbkst;
  FBKST_REQUIRE(A && W && out && partial, "fbkst_linear_argmax_f32: null pointer");
  FBKST_REQUIRE(M > 0 && N > 0 && K > 0 && K % 8 == 0 && lda % 8 == 0 && ldw % 8 == 0 && ldo % 4 == 0 && ldo >= N,
                "fbkst_linear_argmax_f32: bad shape / pitch");
  FBKST_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "fbkst_linear_argmax_f32: out must be 16-byte aligned");
  // (the un-bumped logit of the bump column stays in the running maximum: exact only for a non-negative bump)
  FBKST_REQUIRE(bump_cols == nullptr || bump >= 0.f, "fbkst_linear_argmax_f32: the logit bump must be >= 0");
  return linear_pair_argmax(A, lda, W, ldw, bias, out, ldo, M, N, K, bump_cols, bump, want_sum, partial, m_limit,
                            m_limit_mult, reinterpret_cast<cudaStream_t>(stream));
}
