// Fused self-attention core for the ST encoder (reference: local_attention.py:115-139 with
// LogPenalty conv_transformer_layer.py:22-27): flash-style streaming softmax on tcgen05.
//
//   S_j = Q K_j^T   tcgen05.mma (M128 x N64 x K64), operands K-major in smem (TMA, 128B swizzle),
//                   S double-buffered in TMEM so QK of tile j+1/j+2 runs under the softmax of tile j
//   P_j = softmax   128 threads, one query row each, the 64 scores of the row held in registers:
//                   key-padding mask (last tile only), log-distance penalty from a per-CTA LUT in
//                   log2 domain indexed by (key - query), lazy max (O is rescaled only when the
//                   running max grows by more than 2^8), exp2 in fp32
//   O  += P_j V_j   tcgen05.mma (M128 x N64 x K64), P as bf16 in swizzled smem (double-buffered),
//                   V consumed MN-major straight from its TMA tile
// PERSISTENT: the grid is 2 CTAs per SM; every CTA walks a static, strided list of work items
// (128-query tile, utterance, head) and treats the key tiles of all its items as ONE flattened
// stream, so barrier init, TMEM allocation, the penalty LUT and -- above all -- the TMA latency
// of the first Q/K/V tiles of an item are paid once per CTA instead of once per item (the
// one-CTA-per-item version spent ~45 % of its life in those prologues: profiles/r01a).  The K/V
// rings, the S/P double buffers and all mbarrier phases simply keep counting across items.
//
// Split-KV inside the CTA: the key tiles of an item alternate between two softmax warpgroups, each
// with its own running (max, sum) and its own O accumulator in TMEM (even tiles -> S[0]/P[0]/O[0],
// odd tiles -> S[1]/P[1]/O[1]); the two partial results are merged once per item.  With 2 CTAs per
// SM this puts 16 softmax warps on an SM (4 per scheduler) instead of 8: the one-group version ran
// at 0.4 IPC per scheduler, stalled on fixed-latency dependencies it had too few warps to hide
// (profiles/r01a_ncu_attention.txt).  Registers are capped at 102/thread (2 x 320 threads), so S is
// read from TMEM twice (max pass, exp pass) instead of being held across the O rescale.
//
//   warp 0     TMA producer (Q single-buffered; K 3-stage, V 2-stage rings)
//   warp 1     TMEM allocator + MMA issuer (QK runs two key tiles ahead of PV, across items)
//   warps 2-5  softmax group 0 (even tiles of the CTA's tile stream), TMEM lane quarter = warp % 4
//   warps 6-9  softmax group 1 (odd tiles)
#include <math.h>
#include <stdlib.h>

#include "host_common.h"
#include "ptx.cuh"

namespace fbkst {

constexpr int AT_BM = 128;  // queries per CTA
constexpr int AT_BN = 64;   // keys per tile
constexpr int AT_HD = 64;   // head dim (all reference archs: embed_dim / heads = 64)
constexpr int AT_QB = AT_BM * AT_HD * 2;  // 16 KB
constexpr int AT_KB = AT_BN * AT_HD * 2;  // 8 KB
constexpr int AT_KST = 3, AT_VST = 2;
// shared memory without the penalty LUT (its size depends on L: see attention_smem_bytes)
constexpr int AT_THREADS = 320;
constexpr int AT_SMEM_FIXED = AT_QB + AT_KST * AT_KB + AT_VST * AT_KB + 2 * AT_QB /*P x2*/ +
                              256 /*barriers*/ + 2 * 2 * AT_BM * 4 /*(m, l) exchange*/ +
                              64 * 16 /*item table*/ + 1024 /*align*/;
// penalty LUT (stored negated): entry o <-> (key - query) = o - lut_off, lut_off = nq*128; keys <
// nkv*64.  One copy, read with scalar LDS in explicit batches of 16: four shifted copies would allow
// LDS.128 but cost 32*L bytes (1 CTA/SM beyond L ~ 700) and bought nothing -- the exp pass is bound
// by the MUFU pipe and the MMA round trip, not by shared-memory issue (profiles/r01c).
static inline int attention_lut_floats(int L) {
  return ((L + AT_BM - 1) / AT_BM) * AT_BM + ((L + AT_BN - 1) / AT_BN) * AT_BN;
}
static inline int attention_smem_bytes(int L) { return AT_SMEM_FIXED + 4 * attention_lut_floats(L); }
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kRescaleThreshold = 8.0f;  // log2 units
// Decoupled kernel, one-pass softmax (default; 0 = max pass + exp pass, two TMEM reads of S): log2 units by
// which a row's raw scores may exceed the running reference before it is raised.
#ifndef FBKST_ATTN_ONEPASS
#define FBKST_ATTN_ONEPASS 1
#endif
constexpr float kGrowThreshold = 24.0f;
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// maximum of 32 raw scores held in two 16-register TMEM load groups
__device__ __forceinline__ float raw_max32(const uint32_t (&a)[16], const uint32_t (&b)[16]) {
  float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
  for (int cc = 0; cc < 16; ++cc) {
    m4[cc & 3] = fmaxf(m4[cc & 3], __uint_as_float(a[cc]));
    m4[(cc + 2) & 3] = fmaxf(m4[(cc + 2) & 3], __uint_as_float(b[cc]));
  }
  return fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
}
// the same over the first nv columns only (a = columns 0..15, b = 16..31 of the half); -inf when nv <= 0
__device__ __forceinline__ float raw_max32_masked(const uint32_t (&a)[16], const uint32_t (&b)[16], int nv) {
  float m = -INFINITY;
#pragma unroll
  for (int cc = 0; cc < 16; ++cc) {
    if (cc < nv) m = fmaxf(m, __uint_as_float(a[cc]));
    if (16 + cc < nv) m = fmaxf(m, __uint_as_float(b[cc]));
  }
  return m;
}

// 2^x on the FMA/ALU pipes for part of every row (Cody-Waite range reduction + degree-3 minimax
// polynomial, max rel. error 7.5e-5 -- far below the bf16 rounding of P): the MUFU pipe runs 16 ex2
// per clock and SM, i.e. 512 clocks for a 128x64 tile whose two UMMAs need 256, so with head_dim 64
// the exponentials -- not the tensor pipe -- set the floor.  AT_NPOLY of every 4 register pairs
// take this path (0 = all MUFU).  x is clamped at -126 (2^-126 * p is ~1e-38, i.e. zero in P).
// MEASURED (profiles/r01f_attention_poly_ab.txt): every pair moved off the MUFU makes the kernel
// SLOWER (cfg2 L=375: 61.4 / 63.5 / 65.5 / 67.6 us for 0..3 of 4) -- the softmax warps are bound by
// issue slots and the MMA round trip, not by the MUFU pipe, so the default stays 0.
#ifndef FBKST_ATTN_NPOLY
#define FBKST_ATTN_NPOLY 0
#endif
constexpr int AT_NPOLY = FBKST_ATTN_NPOLY;
__device__ __forceinline__ float2 ex2_poly2(float2 x) {
  const float kMagic = 12582912.0f;  // 1.5 * 2^23: the integer part of x lands in the low mantissa bits
  x.x = fmaxf(x.x, -126.0f);
  x.y = fmaxf(x.y, -126.0f);
  const float2 r = fadd2(x, make_float2(kMagic, kMagic));
  const float2 n = fadd2(r, make_float2(-kMagic, -kMagic));
  const float2 f = ffma2(n, make_float2(-1.0f, -1.0f), x);  // x - round(x) in [-0.5, 0.5]
  float2 p = ffma2(f, make_float2(0.0551716648f, 0.0551716648f), make_float2(0.2426111251f, 0.2426111251f));
  p = ffma2(p, f, make_float2(0.6932609677f, 0.6932609677f));
  p = ffma2(p, f, make_float2(0.9999280572f, 0.9999280572f));
  p.x = __uint_as_float(__float_as_uint(p.x) + (__float_as_uint(r.x) << 23));
  p.y = __uint_as_float(__float_as_uint(p.y) + (__float_as_uint(r.y) << 23));
  return p;
}

// Optional timeline of CTA 0 (debug only; null in production): rows of 16 x int64 per key tile of
// the CTA's stream: [0] MMA: p_full seen  [1] MMA: PV issued  [2] MMA: QK(+2) issued
// [3] softmax: s_full seen  [4] pass 1 done  [5] P/O free  [6] p_full arrive  [7] item epilogue done (last tile row)
// [8] MMA: s_free seen (before QK(+2))  [9] MMA: k_full seen (row = the tile being QK'd)  [10] producer: K issued
// [11] producer: V issued  [12] MMA: v_full seen
// Compiled in only with -DFBKST_ATTN_TRACE (scripts/trace_attn.py); the hooks cost a few percent.
__device__ long long* g_attn_trace = nullptr;
#ifdef FBKST_ATTN_TRACE
#define AT_TRACE(tile, slot)                                                         \
  do {                                                                               \
    if (trace != nullptr && (tile) < 64) trace[(tile) * 16 + (slot)] = clock64();    \
  } while (0)
#else
#define AT_TRACE(tile, slot) \
  do {                       \
  } while (0)
#endif

// Static work list of a CTA: items w = blockIdx.x, blockIdx.x + gridDim.x, ...; item index
// w = (b*H + h)*nq + q_tile, so CTAs running side by side share K/V of one (b, h) through L2.
// The first AT_TABLE items of the CTA are decoded once, cooperatively, into shared memory: the
// integer divisions and the lengths[] load (a global-memory round trip) would otherwise sit on the
// critical path of all three roles at every item boundary.
constexpr int AT_TABLE = 64;
struct AttnItem {
  int w, q0, b, h, len, n_kv;  // n_kv == 0: tile of padded queries (zero fill, no pipeline work)
};
__device__ __forceinline__ int4 attn_decode_raw(int w, const int* __restrict__ lengths, int L, int H,
                                                int nq) {
  const int qt = w % nq, bh = w / nq;
  const int b = bh / H, h = bh - b * H;
  const int q0 = qt * AT_BM;
  const int len = min(__ldg(lengths + b), L);
  return make_int4(q0, b, h, q0 < len ? len : 0);  // length 0: a tile of padded queries
}
struct AttnList {
  const int4* table;  // shared memory
  const int* lengths;
  int L, H, nq, n_items;
  __device__ __forceinline__ void get(AttnItem& it, int k) const {  // k-th item of this CTA
    it.w = blockIdx.x + k * gridDim.x;
    if (it.w >= n_items) return;
    const int4 r = (k < AT_TABLE) ? table[k] : attn_decode_raw(it.w, lengths, L, H, nq);
    it.q0 = r.x;
    it.b = r.y;
    it.h = r.z;
    it.len = r.w;
    // derived here, not packed beside the length: an 8-bit count wraps at 256 key tiles (L > 16320)
    it.n_kv = static_cast<unsigned>(it.len + AT_BN - 1) / AT_BN;
  }
  // next item at or after index k that has pipeline work (n_kv > 0); returns its index
  __device__ __forceinline__ int next_work(AttnItem& it, int k) const {
    for (;; ++k) {
      get(it, k);
      if (it.w >= n_items || it.n_kv > 0) return k;
    }
  }
};

template <int LOGPEN>
__global__ void __launch_bounds__(AT_THREADS, 2)
    attention_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                         __nv_bfloat16* __restrict__ out, const int* __restrict__ lengths, int L, int B,
                         int H, const int* __restrict__ q_limit) {
  const int D = H * AT_HD;
  const int nq = (L + AT_BM - 1) / AT_BM;
  const int n_items = nq * B * H;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
#ifdef FBKST_ATTN_TRACE
  long long* trace = (blockIdx.x == 0 && (lane == 0)) ? g_attn_trace : nullptr;  // lane 0 of each warp
#endif

  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment by pointer arithmetic (keeps the shared address space visible to ptxas)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + AT_QB;            // AT_KST stages
  uint8_t* sV = sK + AT_KST * AT_KB;   // AT_VST stages
  uint8_t* sP = sV + AT_VST * AT_KB;   // 2 x [128 rows x 128 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * AT_QB);
  float* sXch = reinterpret_cast<float*>(bars + 32);  // [group][m | l][128 rows]
  int4* sItems = reinterpret_cast<int4*>(sXch + 2 * 2 * AT_BM);
  float* sLut = reinterpret_cast<float*>(sItems + AT_TABLE);
  uint64_t* q_full = bars + 0;
  uint64_t* k_full = bars + 1;    // [3]
  uint64_t* k_empty = bars + 4;   // [3]
  uint64_t* v_full = bars + 7;    // [2]
  uint64_t* v_empty = bars + 9;   // [2]
  uint64_t* s_full = bars + 11;   // [2]
  uint64_t* p_full = bars + 13;   // [2]
  uint64_t* pv_done = bars + 15;  // [2]
  uint64_t* q_empty = bars + 17;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);
  uint64_t* s_free = bars + 20;   // [2] softmax group -> MMA: S[grp] has been read for the last time

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    mbar_init(q_full, 1);
    mbar_init(q_empty, 1);
    for (int s = 0; s < AT_KST; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&k_empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&v_full[s], 1);
      mbar_init(&v_empty[s], 1);
      mbar_init(&s_full[s], 1);
      mbar_init(&p_full[s], 128);
      mbar_init(&pv_done[s], 1);
      mbar_init(&s_free[s], 128);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 256);
    tmem_relinquish();
  }
  pdl_launch_dependents();
  pdl_wait();  // barrier init / TMEM allocation above overlap the previous kernel's tail
  if (threadIdx.x >= 64 && threadIdx.x < 64 + AT_TABLE) {
    const int w = blockIdx.x + (threadIdx.x - 64) * gridDim.x;
    if (w < n_items) sItems[threadIdx.x - 64] = attn_decode_raw(w, lengths, L, H, nq);
  }
  const AttnList items{sItems, lengths, L, H, nq, n_items};
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_O = tmem_base + 128;  // S[0] +0, S[1] +64, O[0] +128, O[1] +192 (64 columns each)

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    // Whole warp in uniform control flow, one ELECTED lane issues: with `if (lane == 0)` ptxas wraps
    // every UTMALDG / UTCHMMA in a divergence waterfall (ELECT / BRA.U.ANY loop + descriptor
    // rebuild, ~14 instructions per MMA); in uniform code the descriptors sit in uniform registers
    // and the four MMAs of a tile issue back to back.
    {
      // Two cursors over the flattened key-tile stream: K runs two tiles ahead of V.  QK(t+2) is
      // issued while tile t is being soft-maxed, so K(t+2) must not queue behind V(t+1), whose
      // buffer frees only when PV(t-1) has completed (one producer thread, blocking waits).
      AttnItem ki, vi;
      int kk_ = items.next_work(ki, 0), vk_ = items.next_work(vi, 0);
      int kj = 0, vj = 0;
      uint32_t gk = 0, gv = 0, n = 0;  // K / V tiles loaded so far, items whose Q has been loaded
      while (ki.w < n_items || vi.w < n_items) {
        if (ki.w < n_items) {
          const int cq = ki.h * AT_HD, ck = D + cq;
          if (kj == 0) {
            mbar_wait(q_empty, (n & 1) ^ 1);  // every QK of the previous item has completed
            if (elect_one()) {
              mbar_arrive_expect_tx(q_full, AT_QB);
              tma_load_3d(sQ, &tmQ, q_full, cq, ki.b, ki.q0);
            }
            __syncwarp();
            ++n;
          }
          const uint32_t ks = gk % AT_KST;
          mbar_wait(&k_empty[ks], ((gk / AT_KST) & 1) ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&k_full[ks], AT_KB);
            tma_load_3d(sK + ks * AT_KB, &tmKV, &k_full[ks], ck, ki.b, kj * AT_BN);
          }
          __syncwarp();
          AT_TRACE(gk, 10);
          ++gk;
          if (++kj == ki.n_kv) {
            kj = 0;
            kk_ = items.next_work(ki, kk_ + 1);
          }
        }
        if (vi.w < n_items && (gk >= gv + 3 || ki.w >= n_items)) {
          const int cv = 2 * D + vi.h * AT_HD;
          const uint32_t vs = gv & 1;
          mbar_wait(&v_empty[vs], ((gv >> 1) & 1) ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&v_full[vs], AT_KB);
            tma_load_3d(sV + vs * AT_KB, &tmKV, &v_full[vs], cv, vi.b, vj * AT_BN);
          }
          __syncwarp();
          AT_TRACE(gv, 11);
          ++gv;
          if (++vj == vi.n_kv) {
            vj = 0;
            vk_ = items.next_work(vi, vk_ + 1);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (see above)
    {
      constexpr uint32_t IDESC_QK = idesc_bf16_f32(AT_BM, AT_BN, 0, 0);
      constexpr uint32_t IDESC_PV = idesc_bf16_f32(AT_BM, AT_HD, 0, 1);
      const uint64_t qdesc = desc_kmajor_sw128(smem_u32(sQ));
      AttnItem qk, pv;  // two cursors over the same item list: QK runs two key tiles ahead of PV
      int qk_k = items.next_work(qk, 0), pv_k = items.next_work(pv, 0);
      int qk_j = 0, pv_j = 0;
      uint32_t gq = 0, gp = 0, nqk = 0;  // global key-tile counters, items started by QK
      auto issue_qk = [&]() {
        if (qk_j == 0) mbar_wait(q_full, nqk & 1);
        const uint32_t ks = gq % AT_KST;
        mbar_wait(&k_full[ks], (gq / AT_KST) & 1);
        AT_TRACE(gq, 9);
        tc_fence_after();
        const uint64_t kdesc = desc_kmajor_sw128(smem_u32(sK + ks * AT_KB));
        const uint32_t d_tmem = tmem_base + (gq & 1) * AT_BN;
        const bool last = qk_j + 1 == qk.n_kv;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < AT_HD / 16; ++k)
            umma_bf16_ss(d_tmem, qdesc + 2 * k, kdesc + 2 * k, IDESC_QK, k != 0);
          umma_commit(&s_full[gq & 1]);
          umma_commit(&k_empty[ks]);
          if (last) umma_commit(q_empty);  // Q may be overwritten once these MMAs have completed
        }
        __syncwarp();
        ++gq;
        if (++qk_j == qk.n_kv) {
          qk_j = 0;
          ++nqk;
          qk_k = items.next_work(qk, qk_k + 1);
        }
      };
      if (qk.w < n_items) issue_qk();
      if (qk.w < n_items) issue_qk();
      while (pv.w < n_items) {
        const uint32_t pb = gp & 1, ph = (gp >> 1) & 1;
        // QK(gp+2) first: its accumulator S[pb] is free as soon as the group has pulled S(gp) into
        // registers (s_free arrives a quarter into the exp pass), long before P(gp) is complete --
        // the group finds S(gp+2) waiting when it finishes tile gp instead of idling for the
        // PV-issue + QK-issue + MMA round trip (1500 of 4700 cycles per tile: profiles/r01c timeline).
        if (qk.w < n_items) {
          mbar_wait(&s_free[pb], ph);
          AT_TRACE(gp, 8);
          tc_fence_after();
          issue_qk();
        }
        AT_TRACE(gp, 2);
        mbar_wait(&p_full[pb], ph);  // P[pb] in smem, O[pb] rescaled / read out
        AT_TRACE(gp, 0);
        mbar_wait(&v_full[pb], ph);
        AT_TRACE(gp, 12);
        tc_fence_after();
        const uint32_t pa = smem_u32(sP + pb * AT_QB), va = smem_u32(sV + pb * AT_KB);
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < AT_BN / 16; ++kk)
            umma_bf16_ss(tmem_O + pb * AT_HD, desc_kmajor_sw128(pa) + 2 * kk,
                         desc_mnmajor_sw128(va + kk * 2048, AT_KB), IDESC_PV, (pv_j >= 2) || kk != 0);
          umma_commit(&pv_done[pb]);
          umma_commit(&v_empty[pb]);
        }
        __syncwarp();
        AT_TRACE(gp, 1);
        ++gp;
        if (++pv_j == pv.n_kv) {
          pv_j = 0;
          pv_k = items.next_work(pv, pv_k + 1);
        }
      }
    }
  } else {
    // ---- softmax / correction / output: thread <-> (query row, key-tile parity)
    const int grp = (warp - 2) >> 2;       // 0: even tiles, 1: odd tiles of the CTA's tile stream
    const int q = (warp & 3) * 32 + lane;  // row in the tile == TMEM lane
    const int st = threadIdx.x - 64;       // 0..255
    const uint32_t lane_addr = static_cast<uint32_t>((warp & 3) * 32) << 16;
    const uint32_t tS = tmem_base + lane_addr + grp * AT_BN;
    const uint32_t tO = tmem_O + lane_addr + grp * AT_HD;        // this group's accumulator
    const uint32_t tO_other = tmem_O + lane_addr + (grp ^ 1) * AT_HD;
    const int swz = q & 7;
    uint64_t* my_s_full = &s_full[grp];
    uint64_t* my_p_full = &p_full[grp];
    uint64_t* my_pv_done = &pv_done[grp];
    uint8_t* myP = sP + grp * AT_QB + q * 128;
    // Penalty LUT, once per CTA: sLut[o] = -log2(max(1, |o - lut_off|)), (key - query) = o - lut_off
    const int lut_off = nq * AT_BM;
    if (LOGPEN) {
      const int n_lut = lut_off + ((L + AT_BN - 1) / AT_BN) * AT_BN;
      for (int o = st; o < n_lut; o += 256) {
        const int d = abs(o - lut_off);
        sLut[o] = (d > 1) ? -__log2f((float)d) : 0.0f;
      }
      named_bar_sync(1, 256);
    }
    uint32_t g = 0;  // key tiles of the CTA's stream before the current item
    const int q_lim = q_limit ? __ldg(q_limit) : L;  // (after pdl_wait: written by the previous kernel)
    AttnItem it;
    for (int k = 0;; ++k) {
      items.get(it, k);
      if (it.w >= n_items) break;
      const int i = it.q0 + q;
      __nv_bfloat16* orow = out + ((size_t)i * B + it.b) * D + it.h * AT_HD + grp * 32;
      if (it.n_kv == 0) {  // tile of padded queries: defined (finite) output, no pipeline work
        if (i < L && it.q0 < q_lim) {  // tiles at or beyond the caller's row limit are never read: skip
          uint4* op = reinterpret_cast<uint4*>(orow);
#pragma unroll
          for (int j = 0; j < 4; ++j) op[j] = make_uint4(0, 0, 0, 0);
        }
        continue;
      }
      float m_used = -INFINITY, l = 0.0f;
      int cnt = 0;            // tiles this group has folded into O[grp] for this item
      uint32_t last_gg = 0;   // stream index of the group's last tile
      for (int j = (int)((g ^ grp) & 1); j < it.n_kv; j += 2) {
        const uint32_t gg = g + j;  // (gg & 1) == grp
        const uint32_t ph = (gg >> 1) & 1;
        const int k0 = j * AT_BN;
        const int nvalid = min(AT_BN, it.len - k0);
        mbar_wait(my_s_full, ph);
        if (warp == 2 || warp == 6) AT_TRACE(gg, 3);
        tc_fence_after();
        // pass 1: row maximum (S is read again in pass 2: registers are the scarce resource)
        float mx = -INFINITY;
        {
          uint32_t s0[32];
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            tmem_ld32(tS + half * 32, s0);
            tmem_ld_wait();
            if (nvalid == AT_BN) {
              float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
              for (int c = 0; c < 32; ++c) m4[c & 3] = fmaxf(m4[c & 3], __uint_as_float(s0[c]));
              mx = fmaxf(mx, fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])));
            } else {
#pragma unroll
              for (int c = 0; c < 32; ++c)
                if (half * 32 + c < nvalid) mx = fmaxf(mx, __uint_as_float(s0[c]));
            }
          }
        }
        const float m_new = fmaxf(m_used, mx * kLog2e);
        // P[grp] and O[grp] were last used by this group's previous tile (stream index gg - 2)
        if (warp == 2 || warp == 6) AT_TRACE(gg, 4);
        if (gg >= 2) mbar_wait(my_pv_done, ph ^ 1);
        if (warp == 2 || warp == 6) AT_TRACE(gg, 5);
        // lazy rescale: only when some row of the warp grew by more than 2^8 (always at the first tile)
        const bool grow = m_new > m_used + kRescaleThreshold;
        if (__any_sync(0xffffffffu, grow)) {
          const float m_next = grow ? m_new : m_used;
          if (cnt > 0) {
            const float alpha = ex2(m_used - m_next);
            tc_fence_after();
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              uint32_t o0[32];
              tmem_ld32(tO + half * 32, o0);
              tmem_ld_wait();
#pragma unroll
              for (int c = 0; c < 32; ++c) o0[c] = __float_as_uint(__uint_as_float(o0[c]) * alpha);
              tmem_st32(tO + half * 32, o0);
            }
            tmem_st_wait();
            l *= alpha;
          }
          m_used = m_next;
        }
        // pass 2: p = 2^(s*log2e - m - pen2), row sum, bf16 pack -> swizzled K-major P row.
        // Packed fp32 (FFMA2/FADD2): one issue slot per two elements for everything but the MUFU.
        const uint32_t lut_addr = smem_u32(sLut + (lut_off - i) + k0);
        const float2 negm2 = make_float2(-m_used, -m_used);
        const float2 l2e2 = make_float2(kLog2e, kLog2e);
        float2 sm2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
        uint64_t* my_s_free = &s_free[grp];
        {
          // S is pulled in 16-column pieces through two register buffers; a buffer is reloaded as soon
          // as its scores have been turned into exponents' arguments, so the LAST read of S happens a
          // quarter into the pass and the accumulator goes back to the MMA warp right there.
          uint32_t sa[16], sb[16];
          float pn[8];
          tmem_ld16(tS, sa);
          tmem_ld16(tS + 16, sb);
          if (LOGPEN) {
#pragma unroll
            for (int c = 0; c < 8; ++c) pn[c] = lds32(lut_addr + c * 4);
          }
          tmem_ld_wait();
#pragma unroll
          for (int ch = 0; ch < 8; ++ch) {  // 8 columns at a time: registers, not ILP, are scarce
            uint32_t(&s0)[16] = (ch & 2) ? sb : sa;
            const int o = (ch & 1) * 8;
            float2 t[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              float2 add = negm2;
              if (LOGPEN) add = fadd2(negm2, make_float2(pn[2 * c], pn[2 * c + 1]));
              t[c] = ffma2(make_float2(__uint_as_float(s0[o + 2 * c]), __uint_as_float(s0[o + 2 * c + 1])),
                           l2e2, add);
            }
            if (ch == 1 || ch == 3) tmem_ld16(tS + (ch + 3) * 8, s0);  // columns 32.. / 48.. into the freed buffer
            if (LOGPEN && ch < 7) {  // penalties of the next 8 columns fly under the exps
#pragma unroll
              for (int c = 0; c < 8; ++c) pn[c] = lds32(lut_addr + ((ch + 1) * 8 + c) * 4);
            }
            if (ch == 3) {  // all of S(gg) is in registers: hand the accumulator back
              tmem_ld_wait();
              tc_fence_before();
              mbar_arrive(my_s_free);
            }
            if (nvalid != AT_BN) {  // last key tile of the utterance: masked keys -> p = 2^-inf = 0
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                if (ch * 8 + 2 * c >= nvalid) t[c].x = -INFINITY;
                if (ch * 8 + 2 * c + 1 >= nvalid) t[c].y = -INFINITY;
              }
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              if (c < AT_NPOLY) {
                t[c] = ex2_poly2(t[c]);
              } else {
                t[c].x = ex2(t[c].x);
                t[c].y = ex2(t[c].y);
              }
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) sm2[c & 1] = fadd2(sm2[c & 1], t[c]);
            reinterpret_cast<uint4*>(myP)[ch ^ swz] =
                make_uint4(pack_bf16x2(t[0].x, t[0].y), pack_bf16x2(t[1].x, t[1].y),
                           pack_bf16x2(t[2].x, t[2].y), pack_bf16x2(t[3].x, t[3].y));
          }
        }
        l += (sm2[0].x + sm2[0].y) + (sm2[1].x + sm2[1].y);
        tc_fence_before();
        fence_proxy_async_smem();
        mbar_arrive(my_p_full);
        if (warp == 2 || warp == 6) AT_TRACE(gg, 6);
        ++cnt;
        last_gg = gg;
      }
      g += it.n_kv;
      // ---- item epilogue: merge the two groups' partial results
      if (cnt > 0) {
        mbar_wait(my_pv_done, (last_gg >> 1) & 1);  // O[grp] final
        tc_fence_after();
      }
      sXch[(grp * 2 + 0) * AT_BM + q] = m_used;  // -inf when this group had no tile
      sXch[(grp * 2 + 1) * AT_BM + q] = l;
      tc_fence_before();
      named_bar_sync(2, 256);
      tc_fence_after();
      const bool other_has = it.n_kv - cnt > 0;  // item-uniform
      const float m_o = sXch[((grp ^ 1) * 2 + 0) * AT_BM + q];
      const float l_o = sXch[((grp ^ 1) * 2 + 1) * AT_BM + q];
      const float mm = fmaxf(m_used, m_o);            // finite: the item has at least one tile
      const float a_me = (cnt > 0) ? ex2(m_used - mm) : 0.0f;
      const float a_ot = other_has ? ex2(m_o - mm) : 0.0f;
      const float inv = 1.0f / (l * a_me + l_o * a_ot);
      // this group writes output columns [32*grp, 32*grp + 32) of the head
      float acc[32];
      {
        uint32_t o0[32];
        if (cnt > 0) {  // warp-uniform (depends on the item only)
          tmem_ld32(tO + grp * 32, o0);
          tmem_ld_wait();
        }
        const float w = a_me * inv;
#pragma unroll
        for (int c = 0; c < 32; ++c) acc[c] = (cnt > 0) ? __uint_as_float(o0[c]) * w : 0.0f;
        if (other_has) {  // its O buffer is final: the other group waited for it before the barrier
          tmem_ld32(tO_other + grp * 32, o0);
          tmem_ld_wait();
          const float w2 = a_ot * inv;
#pragma unroll
          for (int c = 0; c < 32; ++c) acc[c] = fmaf(__uint_as_float(o0[c]), w2, acc[c]);
        }
      }
      if (i < L) {
        uint4* op = reinterpret_cast<uint4*>(orow);
#pragma unroll
        for (int gq = 0; gq < 4; ++gq) {
          const int o = gq * 8;
          op[gq] = make_uint4(pack_bf16x2(acc[o], acc[o + 1]), pack_bf16x2(acc[o + 2], acc[o + 3]),
                              pack_bf16x2(acc[o + 4], acc[o + 5]), pack_bf16x2(acc[o + 6], acc[o + 7]));
        }
      }
      // both O buffers have been read by both groups before either group lets the MMA warp start
      // the next item's PV (its p_full arrivals come after this barrier)
      tc_fence_before();
      named_bar_sync(3, 256);
      if (warp == 2 || warp == 6) AT_TRACE(g - 1, 7 - 0);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}


// =====================================================================================================
// Decoupled variant (default whenever two of its CTAs fit an SM, i.e. L <~ 1100 with the penalty LUT;
// FBKST_ATTN_DEC=0 forces the split-KV kernel above, which also serves longer L): the two softmax
// warpgroups of a CTA own DIFFERENT work items (group g takes items g, g+2, g+4, ... of the CTA's list)
// instead of the even / odd key tiles of one item.  With split-KV the two groups start every item in
// lock step, the item ends with a cross-group merge (two named barriers, both O buffers read by both
// groups) and the faster group idles until the slower one has finished -- 5-6 k of the 14.5 k cycles
// of an item (profiles/r01g_attention_timeline.txt).  Here a group runs pass 1 / exp pass / its own
// 64-column epilogue back to back and never waits for the other group.  Costs one more Q buffer.
// History (profiles/r01g_attention_decoupled_ab.txt):
//   v1  one in-order thread issuing QK and PV for both groups: parity green, NOT faster (62.5 vs 61.4 us
//       at cfg2) -- the group that finished first waited 1300-1800 cycles for its next S because the
//       thread was blocked on the other group's p_full;
//   v2  (this code) warp 1 issues QK only (blocking, in the fixed interleaved order); warp 0 is an
//       event loop over non-blocking mbarrier.test_wait probes that issues K/Q loads, V loads and PV
//       MMAs as their barriers complete: S-wait 170-250 cycles, 59.5 vs 61.4 us at L=375, ragged cfg3
//       attention 0.644 vs 0.662 ms/step, nothing slower.
//   v3  (round 2) one-pass softmax (ONE TMEM read of S: the row maximum is only an overflow guard because P is
//       bf16 and l / O are fp32, see the tile loop), P and V handed over in two 32-key halves with their own
//       barriers, PV and V streams of the two groups independent of each other: parity green, SAME time
//       (61.4 us) -- and so is the kernel with the LUT loads, the exponentials and the P stores all knocked out
//       (59.4 us).  The softmax arithmetic is not what bounds this kernel.
// What bounds it (profiles/r02y_ncu_attention.txt, r02w_attention_timeline.txt, r02y_umma_probe.txt): 13 % of the
// warp-time sits at the final barrier (1536 items over 592 groups = 2.59 each: one group of most CTAs idles for an
// item), 12 % in the softmax warps' mbarrier waits (next S, the PV halves, the last PV of an item), and the exp pass
// itself issues one instruction per ~10 cycles and warp (short-scoreboard / fixed-latency stalls; 96 registers leave
// no room to pipeline two chunks).  The tensor pipe is not the limiter: an N = 64 tcgen05.mma takes 133 cycles in a
// chain but independent chains overlap to ~53 cycles aggregate, 1700 of the ~3500 cycles of a tile period.  An L2
// prefetch of the next item's boxes and a TMA store of the output tile were measured slower (66.6 / 63.5 us).
constexpr int ATD_SMEM_FIXED = 2 * AT_QB + AT_KST * AT_KB + 2 * AT_KB + 2 * AT_QB /*P x2*/ +
                               256 /*barriers*/ + 64 * 16 /*item table*/ + 1024 /*align*/;
static inline int attention_dec_smem_bytes(int L) { return ATD_SMEM_FIXED + 4 * attention_lut_floats(L); }

// Tile stream of one softmax group: items k = grp, grp + 2, ... of the CTA's list, key tiles in order.
struct GrpCursor {
  AttnItem it;
  int k, j;      // index in the CTA's item list, key tile inside the item
  uint32_t c, n; // tiles / items of this group before the current one
  __device__ __forceinline__ void seek(const AttnList& items) {  // first item at or after k with work
    for (;; k += 2) {
      items.get(it, k);
      if (it.w >= items.n_items || it.n_kv > 0) return;
    }
  }
  __device__ __forceinline__ void init(const AttnList& items, int grp) {
    k = grp; j = 0; c = 0; n = 0;
    seek(items);
  }
  __device__ __forceinline__ bool valid(int n_items) const { return it.w < n_items; }
  __device__ __forceinline__ void advance(const AttnList& items) {
    ++c;
    if (++j == it.n_kv) {
      j = 0; ++n; k += 2;
      seek(items);
    }
  }
};

template <int LOGPEN>
__global__ void __launch_bounds__(AT_THREADS, 2)
    attention_fwd_dec_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                             const __grid_constant__ CUtensorMap tmV, __nv_bfloat16* __restrict__ out, const int* __restrict__ lengths, int L, int B,
                             int H, const int* __restrict__ q_limit) {
  const int D = H * AT_HD;
  const int nq = (L + AT_BM - 1) / AT_BM;
  const int n_items = nq * B * H;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
#ifdef FBKST_ATTN_TRACE
  long long* trace = (blockIdx.x == 0 && (lane == 0)) ? g_attn_trace : nullptr;
#endif
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sQ = smem;                  // 2 x 16 KB: one per group
  uint8_t* sK = sQ + 2 * AT_QB;        // AT_KST stages, shared by both groups (fixed interleaved order)
  uint8_t* sV = sK + AT_KST * AT_KB;   // one per group
  uint8_t* sP = sV + 2 * AT_KB;        // one per group
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * AT_QB);
  int4* sItems = reinterpret_cast<int4*>(bars + 32);
  float* sLut = reinterpret_cast<float*>(sItems + AT_TABLE);
  uint64_t* q_full = bars + 0;    // [2]
  uint64_t* q_empty = bars + 2;   // [2]
  uint64_t* k_full = bars + 4;    // [3]
  uint64_t* k_empty = bars + 7;   // [3]
  // V is loaded in the same two 32-key halves the PV product consumes (boxes of tmV), each half free again as
  // soon as ITS PV half has completed (pv_lo / pv_hi): the next tile's V is on its way half a tile before it is
  // needed, although V is single-buffered
  uint64_t* v_lo = bars + 10;     // [2]
  uint64_t* v_hi = bars + 12;     // [2]
  uint64_t* s_full = bars + 14;   // [2]
  // P is handed to the tensor pipe in two 32-key halves (same 16 KB tile, k-steps 0-1 / 2-3 of the PV product),
  // each with its own full / done barrier: the first half of the NEXT tile's P only waits for the PV half that
  // was issued half a tile earlier, so the one-pass softmax never sits on the latency of the PV it just requested
  uint64_t* p_lo = bars + 16;     // [2]
  uint64_t* pv_lo = bars + 18;    // [2]
  uint64_t* s_free = bars + 20;   // [2]
  uint64_t* p_hi = bars + 22;     // [2]
  uint64_t* pv_hi = bars + 24;    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 26);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmKV);
    tma_prefetch_desc(&tmV);
    for (int s = 0; s < AT_KST; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&k_empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&q_full[s], 1);
      mbar_init(&q_empty[s], 1);
      mbar_init(&v_lo[s], 1);
      mbar_init(&v_hi[s], 1);
      mbar_init(&s_full[s], 1);
      mbar_init(&p_lo[s], 128);
      mbar_init(&p_hi[s], 128);
      mbar_init(&pv_lo[s], 1);
      mbar_init(&pv_hi[s], 1);
      mbar_init(&s_free[s], 128);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 256);
    tmem_relinquish();
  }
  pdl_launch_dependents();
  pdl_wait();
  if (threadIdx.x >= 64 && threadIdx.x < 64 + AT_TABLE) {
    const int w = blockIdx.x + (threadIdx.x - 64) * gridDim.x;
    if (w < n_items) sItems[threadIdx.x - 64] = attn_decode_raw(w, lengths, L, H, nq);
  }
  const AttnList items{sItems, lengths, L, H, nq, n_items};
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_O = tmem_base + 128;  // S[0] +0, S[1] +64, O[0] +128, O[1] +192

  // Fixed interleaved order of the two groups' tile streams (identical in the TMA warp and the MMA
  // warp): take the group whose turn it is, or the other one when that stream is exhausted; the turn
  // flips after every tile.
#define ATD_PICK(c0, c1, turn) (((turn) == 0) ? ((c0).valid(n_items) ? 0 : 1) : ((c1).valid(n_items) ? 1 : 0))

  if (warp == 0) {
    // ---------------------------------------------- TMA loads (Q, K, V) + PV issue, EVENT DRIVEN
    // Three cursors walk the fixed interleaved order (K loads, V loads, PV issues); each step is taken
    // as soon as ITS barrier(s) have completed (non-blocking test_wait), so a PV never queues behind a
    // K load whose ring slot is still busy and vice versa.  The QK issuer (warp 1) has the blocking,
    // strictly ordered waits.  (FBKST_ATTN_DEC: with one in-order thread issuing both QK and PV the
    // group that finished its tile first waited for the other group's p_full before its next S was
    // even requested: 1300-1800 of 4000 cycles per tile, profiles/r01g_attention_decoupled_ab.txt.)
    constexpr uint32_t IDESC_PV = idesc_bf16_f32(AT_BM, AT_HD, 0, 1);
    GrpCursor kc0, kc1, vc0, vc1, pc0, pc1;
    kc0.init(items, 0); kc1.init(items, 1); vc0.init(items, 0); vc1.init(items, 1);
    pc0.init(items, 0); pc1.init(items, 1);
    int kturn = 0;
    uint32_t gk = 0;
    auto try_k = [&](GrpCursor& c, int g) -> bool {
      const uint32_t ks = gk % AT_KST;
      if (!mbar_test_wait(&k_empty[ks], ((gk / AT_KST) & 1) ^ 1)) return false;
      if (c.j == 0 && !mbar_test_wait(&q_empty[g], (c.n & 1) ^ 1)) return false;
      const int cq = c.it.h * AT_HD, ck = D + cq;
      if (elect_one()) {
        if (c.j == 0) {
          mbar_arrive_expect_tx(&q_full[g], AT_QB);
          tma_load_3d(sQ + g * AT_QB, &tmQ, &q_full[g], cq, c.it.b, c.it.q0);
        }
        mbar_arrive_expect_tx(&k_full[ks], AT_KB);
        tma_load_3d(sK + ks * AT_KB, &tmKV, &k_full[ks], ck, c.it.b, c.j * AT_BN);
      }
      __syncwarp();
      ++gk;
      c.advance(items);
      return true;
    };
    int v_half[2] = {0, 0};  // which half of the group's current V tile is loaded next
    auto try_v = [&](GrpCursor& c, int g) -> bool {
      const int hf = v_half[g];
      // the half-buffer was read by the matching PV half of the group's previous tile
      if (c.c >= 1 && !mbar_test_wait(hf ? &pv_hi[g] : &pv_lo[g], (c.c - 1) & 1)) return false;
      const int cv = 2 * D + c.it.h * AT_HD;
      if (elect_one()) {
        uint64_t* bar = hf ? &v_hi[g] : &v_lo[g];
        mbar_arrive_expect_tx(bar, AT_KB / 2);
        tma_load_3d(sV + g * AT_KB + hf * (AT_KB / 2), &tmV, bar, cv, c.it.b, c.j * AT_BN + hf * (AT_BN / 2));
      }
      __syncwarp();
      v_half[g] = hf ^ 1;
      if (hf == 1) c.advance(items);
      return true;
    };
    int pv_half[2] = {0, 0};  // which half of the group's current tile is issued next
    auto try_pv = [&](GrpCursor& c, int g) -> bool {
      const uint32_t ph = c.c & 1;
      const int hf = pv_half[g];
      if (hf == 0) {
        if (!mbar_test_wait(&p_lo[g], ph) || !mbar_test_wait(&v_lo[g], ph)) return false;
      } else {
        if (!mbar_test_wait(&p_hi[g], ph) || !mbar_test_wait(&v_hi[g], ph)) return false;
      }
      tc_fence_after();
      const uint32_t pa = smem_u32(sP + g * AT_QB), va = smem_u32(sV + g * AT_KB);
      if (elect_one()) {
#pragma unroll
        for (int k2 = 0; k2 < 2; ++k2) {
          const int kk = hf * 2 + k2;
          umma_bf16_ss(tmem_O + g * AT_HD, desc_kmajor_sw128(pa) + 2 * kk,
                       desc_mnmajor_sw128(va + kk * 2048, AT_KB), IDESC_PV, (c.j > 0) || kk != 0);
        }
        umma_commit(hf ? &pv_hi[g] : &pv_lo[g]);
      }
      __syncwarp();
      pv_half[g] = hf ^ 1;
      if (hf == 1) c.advance(items);
      return true;
    };
    uint32_t idle = 0;
    for (;;) {
      const bool k_left = kc0.valid(n_items) || kc1.valid(n_items);
      const bool v_left = vc0.valid(n_items) || vc1.valid(n_items);
      const bool p_left = pc0.valid(n_items) || pc1.valid(n_items);
      if (!k_left && !v_left && !p_left) break;
      bool progressed = false;
      if (p_left) {  // PV first: it is what the softmax groups wait for; the groups' PV streams are independent
        if (pc0.valid(n_items) && try_pv(pc0, 0)) progressed = true;
        if (pc1.valid(n_items) && try_pv(pc1, 1)) progressed = true;
      }
      if (k_left) {
        const bool ok = (ATD_PICK(kc0, kc1, kturn) == 0) ? try_k(kc0, 0) : try_k(kc1, 1);
        if (ok) { kturn ^= 1; progressed = true; }
      }
      if (v_left) {  // per-group buffers: the groups' V streams are independent as well
        if (vc0.valid(n_items) && try_v(vc0, 0)) progressed = true;
        if (vc1.valid(n_items) && try_v(vc1, 1)) progressed = true;
      }
      if (!progressed) __nanosleep(32);  // do not take issue slots from the softmax warps of this SMSP
#if FBKST_WATCHDOG
      idle = progressed ? 0 : idle + 1;
      if (idle > (1u << 27)) {
        printf("fbkst: attention event loop watchdog block=%d\n", blockIdx.x);
        __trap();
      }
#endif
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ QK issuer (blocking, in order)
    constexpr uint32_t IDESC_QK = idesc_bf16_f32(AT_BM, AT_BN, 0, 0);
    GrpCursor qc0, qc1;
    qc0.init(items, 0); qc1.init(items, 1);
    int qturn = 0;
    uint32_t gq = 0;
    auto issue_qk = [&](GrpCursor& c, int g) {
      if (c.c >= 1) {  // S[g] must have been pulled into registers by the group's previous tile
        mbar_wait(&s_free[g], (c.c - 1) & 1);
      }
      if (c.j == 0) mbar_wait(&q_full[g], c.n & 1);
      const uint32_t ks = gq % AT_KST;
      mbar_wait(&k_full[ks], (gq / AT_KST) & 1);
      tc_fence_after();
      const uint64_t qdesc = desc_kmajor_sw128(smem_u32(sQ + g * AT_QB));
      const uint64_t kdesc = desc_kmajor_sw128(smem_u32(sK + ks * AT_KB));
      const uint32_t d_tmem = tmem_base + g * AT_BN;
      const bool last = c.j + 1 == c.it.n_kv;
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < AT_HD / 16; ++k)
          umma_bf16_ss(d_tmem, qdesc + 2 * k, kdesc + 2 * k, IDESC_QK, k != 0);
        umma_commit(&s_full[g]);
        umma_commit(&k_empty[ks]);
        if (last) umma_commit(&q_empty[g]);  // Q[g] may be overwritten once these MMAs have completed
      }
      __syncwarp();
      ++gq;
      c.advance(items);
    };
    while (qc0.valid(n_items) || qc1.valid(n_items)) {
      if (ATD_PICK(qc0, qc1, qturn) == 0) issue_qk(qc0, 0); else issue_qk(qc1, 1);
      qturn ^= 1;
    }
  } else {
    // ---- softmax / correction / output: thread <-> (query row of the group's own item)
    const int grp = (warp - 2) >> 2;
    const int q = (warp & 3) * 32 + lane;  // row in the tile == TMEM lane
    const int st = threadIdx.x - 64;       // 0..255
    const uint32_t lane_addr = static_cast<uint32_t>((warp & 3) * 32) << 16;
    const uint32_t tS = tmem_base + lane_addr + grp * AT_BN;
    const uint32_t tO = tmem_O + lane_addr + grp * AT_HD;
    const int swz = q & 7;
    uint64_t* my_s_full = &s_full[grp];
    uint64_t* my_p_lo = &p_lo[grp];
    uint64_t* my_p_hi = &p_hi[grp];
    uint64_t* my_pv_lo = &pv_lo[grp];
    uint64_t* my_pv_hi = &pv_hi[grp];
    uint64_t* my_s_free = &s_free[grp];
    uint8_t* myP = sP + grp * AT_QB + q * 128;
    const int lut_off = nq * AT_BM;
    if (LOGPEN) {
      const int n_lut = lut_off + ((L + AT_BN - 1) / AT_BN) * AT_BN;
      for (int o = st; o < n_lut; o += 256) {
        const int d = abs(o - lut_off);
        sLut[o] = (d > 1) ? -__log2f((float)d) : 0.0f;
      }
      named_bar_sync(1, 256);
    }
    uint32_t c = 0;  // key tiles of this group before the current one
    const int q_lim = q_limit ? __ldg(q_limit) : L;  // (after pdl_wait: written by the previous kernel)
    AttnItem it;
    for (int k = grp;; k += 2) {
      items.get(it, k);
      if (it.w >= n_items) break;
      const int i = it.q0 + q;
      __nv_bfloat16* orow = out + ((size_t)i * B + it.b) * D + it.h * AT_HD;
      if (it.n_kv == 0) {  // tile of padded queries: defined (finite) output, no pipeline work
        if (i < L && it.q0 < q_lim) {  // tiles at or beyond the caller's row limit are never read: skip
          uint4* op = reinterpret_cast<uint4*>(orow);
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) op[jj] = make_uint4(0, 0, 0, 0);
        }
        continue;
      }
      float m_used = -INFINITY, l = 0.0f;
      for (int j = 0; j < it.n_kv; ++j, ++c) {
        const uint32_t ph = c & 1;
        const int k0 = j * AT_BN;
        const int nvalid = min(AT_BN, it.len - k0);
        mbar_wait(my_s_full, ph);
        if (warp == 2 || warp == 6) AT_TRACE(2 * c + grp, 3);
        tc_fence_after();
#if FBKST_ATTN_ONEPASS
        // ONE pass over S (one TMEM read): the row maximum is only an overflow guard here -- P is bf16 and
        // l / O are fp32, all with the fp32 exponent range, so any reference m_used within 2^kGrowThreshold
        // of the row's scores gives the same softmax.  The raw maximum of each 32-column half is taken from
        // the registers the half was loaded into, BEFORE S is handed back: the first half may raise the
        // reference (always at an item's first tile), a second half that exceeds it restarts the tile
        // (S is still in TMEM) -- rare: scores 16.6 nats above everything the row has seen so far.
        const uint32_t lut_addr = smem_u32(sLut + (lut_off - i) + k0);
        const float2 l2e2 = make_float2(kLog2e, kLog2e);
        float2 sm2[2];
        float m_restart = -INFINITY;  // reference demanded by a second half that overflowed (restart)
        for (;;) {
          uint32_t sa[16], sb[16];
          float pn[8];
          bool redo = false;
          tmem_ld16(tS, sa);
          tmem_ld16(tS + 16, sb);
          if (LOGPEN) {
#pragma unroll
            for (int cc = 0; cc < 8; ++cc) pn[cc] = lds32(lut_addr + cc * 4);
          }
          sm2[0] = make_float2(0.f, 0.f);
          sm2[1] = make_float2(0.f, 0.f);
          tmem_ld_wait();
          if (warp == 2 || warp == 6) AT_TRACE(2 * c + grp, 8);
          {
            const float m_half =
                fmaxf((nvalid == AT_BN ? raw_max32(sa, sb) : raw_max32_masked(sa, sb, nvalid)) * kLog2e, m_restart);
            const bool grow = m_half > m_used + kGrowThreshold;
            if (__any_sync(0xffffffffu, grow)) {
              const float m_next = grow ? m_half : m_used;
              if (j > 0) {
                mbar_wait(my_pv_hi, ph ^ 1);  // O[grp] quiescent: every PV of the previous tile has completed
                const float alpha = ex2(m_used - m_next);
                tc_fence_after();
                // rare path: rolled, 8 columns at a time, so that it costs the hot path no registers
#pragma unroll 1
                for (int cb = 0; cb < AT_HD; cb += 8) {
                  uint32_t o0[8];
                  tmem_ld8(tO + cb, o0);
                  tmem_ld_wait();
#pragma unroll
                  for (int cc = 0; cc < 8; ++cc) o0[cc] = __float_as_uint(__uint_as_float(o0[cc]) * alpha);
                  tmem_st8(tO + cb, o0);
                }
                tmem_st_wait();
                l *= alpha;
              }
              m_used = m_next;
            }
          }
          if (warp == 2 || warp == 6) AT_TRACE(2 * c + grp, 4);
          const float2 negm2 = make_float2(-m_used, -m_used);
#pragma unroll
          for (int ch = 0; ch < 8; ++ch) {
            uint32_t(&s0)[16] = (ch & 2) ? sb : sa;
            const int o = (ch & 1) * 8;
            float2 t[4];
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
              float2 add = negm2;
              if (LOGPEN) add = fadd2(negm2, make_float2(pn[2 * cc], pn[2 * cc + 1]));
              t[cc] = ffma2(make_float2(__uint_as_float(s0[o + 2 * cc]), __uint_as_float(s0[o + 2 * cc + 1])),
                            l2e2, add);
            }
            if (ch == 1 || ch == 3) tmem_ld16(tS + (ch + 3) * 8, s0);
            if (LOGPEN && ch < 7) {
#pragma unroll
              for (int cc = 0; cc < 8; ++cc) pn[cc] = lds32(lut_addr + ((ch + 1) * 8 + cc) * 4);
            }
            if (ch == 3) {  // the second half is in registers: check it, then hand the accumulator back
              tmem_ld_wait();
              if (warp == 2 || warp == 6) AT_TRACE(2 * c + grp, 9);
              const float m_half =
                  (nvalid == AT_BN ? raw_max32(sa, sb) : raw_max32_masked(sa, sb, nvalid - 32)) * kLog2e;
              const bool grow = m_half > m_used + kGrowThreshold;
              if (__any_sync(0xffffffffu, grow)) {
                // restart the tile against the raised reference (the first-half path rescales O / l)
                redo = true;
                m_restart = grow ? m_half : -INFINITY;
                break;
              }
              tc_fence_before();
              mbar_arrive(my_s_free);
              if (warp == 2 || warp == 6) AT_TRACE(2 * c + grp, 10);
            }
            if (nvalid != AT_BN) {
#pragma unroll
              for (int cc = 0; cc < 4; ++cc) {
                if (ch * 8 + 2 * cc >= nvalid) t[cc].x = -INFINITY;
                if (ch * 8 + 2 * cc + 1 >= nvalid) t[cc].y = -INFINITY;
              }
            }
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
              t[cc].x = ex2(t[cc].x);
              t[cc].y = ex2(t[cc].y);
            }
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) sm2[cc & 1] = fadd2(sm2[cc & 1], t[cc]);
            // the half of P[grp] about to be overwritten was read by the matching PV half of the previous tile
            if (ch == 0 && c >= 1) mbar_wait(my_pv_lo, ph ^ 1);
            if (ch == 4 && c >= 1) mbar_wait(my_pv_hi, ph ^ 1);
            if (ch == 4 && (warp == 2 || warp == 6)) AT_TRACE(2 * c + grp, 12);
            if (ch == 0 && (warp == 2 || warp == 6)) AT_TRACE(2 * c + grp, 5);
            reinterpret_cast<uint4*>(myP)[ch ^ swz] =
                make_uint4(pack_bf16x2(t[0].x, t[0].y), pack_bf16x2(t[1].x, t[1].y),
                           pack_bf16x2(t[2].x, t[2].y), pack_bf16x2(t[3].x, t[3].y));
            if (ch == 3) {
              tc_fence_before();  // (orders the O reads of the previous item's epilogue / a rescale before PV)
              fence_proxy_async_smem();
              mbar_arrive(my_p_lo);
              if (warp == 2 || warp == 6) AT_TRACE(2 * c + grp, 11);
            }
          }
          if (!redo) break;
        }
#else
        // pass 1: row maximum (S is read again in pass 2: registers are the scarce resource)
        float mx = -INFINITY;
        {
          uint32_t s0[32];
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            tmem_ld32(tS + half * 32, s0);
            tmem_ld_wait();
            if (nvalid == AT_BN) {
              float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
              for (int cc = 0; cc < 32; ++cc) m4[cc & 3] = fmaxf(m4[cc & 3], __uint_as_float(s0[cc]));
              mx = fmaxf(mx, fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])));
            } else {
#pragma unroll
              for (int cc = 0; cc < 32; ++cc)
                if (half * 32 + cc < nvalid) mx = fmaxf(mx, __uint_as_float(s0[cc]));
            }
          }
        }
        const float m_new = fmaxf(m_used, mx * kLog2e);
        if (warp == 2 || warp == 6) AT_TRACE(2 * c + grp, 4);
        // P[grp] / O[grp] were last used by this group's previous tile
        if (c >= 1) mbar_wait(my_pv_hi, ph ^ 1);
        if (warp == 2 || warp == 6) AT_TRACE(2 * c + grp, 5);
        const bool grow = m_new > m_used + kRescaleThreshold;
        if (__any_sync(0xffffffffu, grow)) {
          const float m_next = grow ? m_new : m_used;
          if (j > 0) {
            const float alpha = ex2(m_used - m_next);
            tc_fence_after();
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              uint32_t o0[32];
              tmem_ld32(tO + half * 32, o0);
              tmem_ld_wait();
#pragma unroll
              for (int cc = 0; cc < 32; ++cc) o0[cc] = __float_as_uint(__uint_as_float(o0[cc]) * alpha);
              tmem_st32(tO + half * 32, o0);
            }
            tmem_st_wait();
            l *= alpha;
          }
          m_used = m_next;
        }
        // pass 2 (same as the split-KV kernel): p = 2^(s*log2e - m - pen2), row sum, bf16 pack
        const uint32_t lut_addr = smem_u32(sLut + (lut_off - i) + k0);
        const float2 negm2 = make_float2(-m_used, -m_used);
        const float2 l2e2 = make_float2(kLog2e, kLog2e);
        float2 sm2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
        {
          uint32_t sa[16], sb[16];
          float pn[8];
          tmem_ld16(tS, sa);
          tmem_ld16(tS + 16, sb);
          if (LOGPEN) {
#pragma unroll
            for (int cc = 0; cc < 8; ++cc) pn[cc] = lds32(lut_addr + cc * 4);
          }
          tmem_ld_wait();
#pragma unroll
          for (int ch = 0; ch < 8; ++ch) {
            uint32_t(&s0)[16] = (ch & 2) ? sb : sa;
            const int o = (ch & 1) * 8;
            float2 t[4];
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
              float2 add = negm2;
              if (LOGPEN) add = fadd2(negm2, make_float2(pn[2 * cc], pn[2 * cc + 1]));
              t[cc] = ffma2(make_float2(__uint_as_float(s0[o + 2 * cc]), __uint_as_float(s0[o + 2 * cc + 1])),
                            l2e2, add);
            }
            if (ch == 1 || ch == 3) tmem_ld16(tS + (ch + 3) * 8, s0);
            if (LOGPEN && ch < 7) {
#pragma unroll
              for (int cc = 0; cc < 8; ++cc) pn[cc] = lds32(lut_addr + ((ch + 1) * 8 + cc) * 4);
            }
            if (ch == 3) {  // all of S is in registers: hand the accumulator back
              tmem_ld_wait();
              tc_fence_before();
              mbar_arrive(my_s_free);
            }
            if (nvalid != AT_BN) {
#pragma unroll
              for (int cc = 0; cc < 4; ++cc) {
                if (ch * 8 + 2 * cc >= nvalid) t[cc].x = -INFINITY;
                if (ch * 8 + 2 * cc + 1 >= nvalid) t[cc].y = -INFINITY;
              }
            }
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
              t[cc].x = ex2(t[cc].x);
              t[cc].y = ex2(t[cc].y);
            }
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) sm2[cc & 1] = fadd2(sm2[cc & 1], t[cc]);
            reinterpret_cast<uint4*>(myP)[ch ^ swz] =
                make_uint4(pack_bf16x2(t[0].x, t[0].y), pack_bf16x2(t[1].x, t[1].y),
                           pack_bf16x2(t[2].x, t[2].y), pack_bf16x2(t[3].x, t[3].y));
          }
        }
#endif
        l += (sm2[0].x + sm2[0].y) + (sm2[1].x + sm2[1].y);
        if (warp == 2 || warp == 6) AT_TRACE(2 * c + grp, 0);
        tc_fence_before();
        fence_proxy_async_smem();
#if !FBKST_ATTN_ONEPASS
        mbar_arrive(my_p_lo);
#endif
        mbar_arrive(my_p_hi);
        if (warp == 2 || warp == 6) AT_TRACE(2 * c + grp, 6);
      }
      // ---- item epilogue (this group only): O / l -> bf16, 128 B per query row.  (Staging the tile in P[grp]
      // and storing it with one TMA box was measured slower: 63.5 vs 62.1 us at cfg2 -- the item boundary is
      // bound by the completion of the last PV, not by these stores.)
      mbar_wait(my_pv_hi, (c - 1) & 1);  // O[grp] final
      tc_fence_after();
      const float inv = 1.0f / l;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t o0[32];
        tmem_ld32(tO + half * 32, o0);
        tmem_ld_wait();
        if (i < L) {
          uint4* op = reinterpret_cast<uint4*>(orow + half * 32);
#pragma unroll
          for (int gq4 = 0; gq4 < 4; ++gq4) {
            const int o = gq4 * 8;
            op[gq4] = make_uint4(
                pack_bf16x2(__uint_as_float(o0[o]) * inv, __uint_as_float(o0[o + 1]) * inv),
                pack_bf16x2(__uint_as_float(o0[o + 2]) * inv, __uint_as_float(o0[o + 3]) * inv),
                pack_bf16x2(__uint_as_float(o0[o + 4]) * inv, __uint_as_float(o0[o + 5]) * inv),
                pack_bf16x2(__uint_as_float(o0[o + 6]) * inv, __uint_as_float(o0[o + 7]) * inv));
          }
        }
      }
      // O[grp] is overwritten by the PV of the group's next tile, which waits for this group's next
      // p_lo arrival (ordered after the TMEM reads above by the fence before that arrive)
      if (warp == 2 || warp == 6) AT_TRACE(2 * (c - 1) + grp, 7);
    }
  }
#undef ATD_PICK
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

}  // namespace fbkst

// debug hook (not part of the public ABI): buffer of 64*8 int64, or NULL to disable
extern "C" int fbkst_debug_set_attention_trace(long long* buf) {
  cudaError_t e = cudaMemcpyToSymbol(fbkst::g_attn_trace, &buf, sizeof(buf));
  return e == cudaSuccess ? 0 : -2;
}

using namespace fbkst;

namespace fbkst {
// attention_wide.cu: one CTA per SM, 128-key tiles; returns 1 when the shape is not served
int attention_wide_launch(const void* qkv, void* out, const int32_t* lengths, int L, int B, int H, int log_penalty,
                          const int32_t* q_limit, cudaStream_t st);
}  // namespace fbkst

static int attention_entry(const void* qkv, void* out, const int32_t* lengths, int L, int B, int H,
                           int log_penalty, const int32_t* q_limit, fbkst_stream_t stream) {
  FBKST_REQUIRE(qkv && out && lengths, "fbkst_attention_fwd: null pointer");
  FBKST_REQUIRE(L > 0 && B > 0 && H > 0, "fbkst_attention_fwd: bad shape L=%d B=%d H=%d", L, B, H);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int D = H * AT_HD;
  // wide kernel (attention_wide.cu: one CTA per SM, 128-key tiles, P through tensor memory) whenever its shared
  // memory fits (L <~ 2500 with the penalty LUT); FBKST_ATTN_WIDE=0 selects the round-1 kernels below (A/B switch)
  static const bool wide_enabled = !(getenv("FBKST_ATTN_WIDE") && atoi(getenv("FBKST_ATTN_WIDE")) == 0);
  if (wide_enabled) {
    const int rc = attention_wide_launch(qkv, out, lengths, L, B, H, log_penalty, q_limit, st);
    if (rc != 1) return rc;
  }
  CUtensorMap tmQ, tmKV, tmV;
  uint64_t dims[3] = {(uint64_t)3 * D, (uint64_t)B, (uint64_t)L};
  uint64_t strides[2] = {(uint64_t)3 * D * 2, (uint64_t)B * 3 * D * 2};
  uint32_t boxq[3] = {AT_HD, 1, AT_BM};
  uint32_t boxk[3] = {AT_HD, 1, AT_BN};
  int rc = make_tensor_map(&tmQ, qkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 3, dims, strides, boxq,
                           nullptr);
  if (rc) return rc;
  rc = make_tensor_map(&tmKV, qkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 3, dims, strides, boxk, nullptr);
  if (rc) return rc;
  uint32_t boxv[3] = {AT_HD, 1, AT_BN / 2};  // V halves of the decoupled kernel
  rc = make_tensor_map(&tmV, qkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 3, dims, strides, boxv, nullptr);
  if (rc) return rc;
  static PerDeviceFlag configured;
  if (!configured) {
    FBKST_CHECK_CUDA(cudaFuncSetAttribute(attention_fwd_kernel<0>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    FBKST_CHECK_CUDA(cudaFuncSetAttribute(attention_fwd_kernel<1>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    FBKST_CHECK_CUDA(cudaFuncSetAttribute(attention_fwd_dec_kernel<0>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    FBKST_CHECK_CUDA(cudaFuncSetAttribute(attention_fwd_dec_kernel<1>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    configured = true;
  }
  // decoupled groups (one item per softmax group) whenever two of its CTAs fit an SM (L <~ 1100 with the
  // penalty LUT); FBKST_ATTN_DEC=0 forces the split-KV kernel (A/B switch)
  static const bool dec_enabled = !(getenv("FBKST_ATTN_DEC") && atoi(getenv("FBKST_ATTN_DEC")) == 0);
  const int smem_dec = attention_dec_smem_bytes(log_penalty ? L : 0);
  const long long n_items_all = (long long)((L + AT_BM - 1) / AT_BM) * B * H;
  if (dec_enabled && 2 * (smem_dec + 1024) <= 228 * 1024) {
    FBKST_REQUIRE(n_items_all < (1ll << 30), "fbkst_attention_fwd: too many work items");
    int grid = num_sms() * 2;
    if (grid > n_items_all) grid = (int)n_items_all;
    if (log_penalty)
      FBKST_CHECK_CUDA(launch_pdl(attention_fwd_dec_kernel<1>, dim3(grid), dim3(AT_THREADS), smem_dec, st,
                                  tmQ, tmKV, tmV, (__nv_bfloat16*)out, lengths, L, B, H, q_limit));
    else
      FBKST_CHECK_CUDA(launch_pdl(attention_fwd_dec_kernel<0>, dim3(grid), dim3(AT_THREADS), smem_dec, st,
                                  tmQ, tmKV, tmV, (__nv_bfloat16*)out, lengths, L, B, H, q_limit));
    return FBKST_OK;
  }
  const int smem = attention_smem_bytes(log_penalty ? L : 0);
  FBKST_REQUIRE(smem <= 227 * 1024, "fbkst_attention_fwd: L=%d needs %d B of shared memory", L, smem);
  // persistent grid: as many CTAs as fit (2 per SM up to L ~ 3000), never more than work items
  const int per_sm = (2 * (smem + 1024) <= 228 * 1024) ? 2 : 1;
  const long long n_items = (long long)((L + AT_BM - 1) / AT_BM) * B * H;
  FBKST_REQUIRE(n_items < (1ll << 31), "fbkst_attention_fwd: too many work items");
  int grid = num_sms() * per_sm;
  if (grid > n_items) grid = (int)n_items;
  if (log_penalty)
    FBKST_CHECK_CUDA(launch_pdl(attention_fwd_kernel<1>, dim3(grid), dim3(AT_THREADS), smem, st, tmQ, tmKV,
                                (__nv_bfloat16*)out, lengths, L, B, H, q_limit));
  else
    FBKST_CHECK_CUDA(launch_pdl(attention_fwd_kernel<0>, dim3(grid), dim3(AT_THREADS), smem, st, tmQ, tmKV,
                                (__nv_bfloat16*)out, lengths, L, B, H, q_limit));
  return FBKST_OK;
}

extern "C" int fbkst_attention_fwd(const void* qkv, void* out, const int32_t* lengths, int L, int B,
                                   int H, int log_penalty, fbkst_stream_t stream) {
  return attention_entry(qkv, out, lengths, L, B, H, log_penalty, nullptr, stream);
}

extern "C" int fbkst_attention_fwd_limited(const void* qkv, void* out, const int32_t* lengths, int L, int B,
                                           int H, int log_penalty, const int32_t* q_limit,
                                           fbkst_stream_t stream) {
  FBKST_REQUIRE(q_limit != nullptr, "fbkst_attention_fwd_limited: null q_limit");
  return attention_entry(qkv, out, lengths, L, B, H, log_penalty, q_limit, stream);
}
