// Self-attention core, "wide" layout: the kernel for every L without the penalty and for L <= 2560 with it
// (reference: local_attention.py:115-139 with LogPenalty conv_transformer_layer.py:22-27); longer inputs with the
// penalty go to the split-KV kernel of attention_tcgen05.cu.  Same arithmetic and the same pipeline roles as the
// round-1 decoupled kernel it replaced (since removed), re-cut for what that kernel's profile showed
// (profiles/r02y_ncu_attention.txt): softmax warps at 7.3 issued instructions per score and ~0.1 IPC each
// (96 registers: one 8-score chunk in flight), 64 KB of P written to and read back from shared memory per
// 128 x 128 scores next to 64 KB of penalty loads on a 128 B/clk path, and 16 M128 x N64 tensor instructions
// per 128 x 128 scores at 133 cycles apiece.
//
//   * ONE CTA per SM, 384 threads: a producer warpgroup that shrinks to 56 registers (warp 0 TMA loads,
//     warp 1 QK issue, warps 2 / 3 PV issue of group 0 / 1) and two softmax warpgroups that grow to 224,
//     each working on its OWN work item (128-query tile, utterance, head);
//   * 128-key tiles: S = Q K^T is ONE chain of four M128 x N128 x K16 instructions per 128 keys;
//     TMEM: S0 | S1 (128 columns each) | O0 | O1 (64) | P0 | P1 (64) = all 512 columns; shared memory:
//     Q x2, K x3, V x2 tiles of 16 KB + 2 x 16 KB of output staging + the LUT = 167 KB + 16 B per LUT entry
//     (L <~ 2400 with the penalty);
//   * the softmax thread (one query row) pulls its whole 128-score row into registers and hands S[g] back at
//     once, so the next QK product runs under this tile's exponentials; key padding is written into the
//     score registers (-inf), after which every tile runs ONE straight-line block of 16 chunks with no
//     shared-memory store inside it (ptxas does not move a chunk's LUT loads above an earlier store), in
//     which the LDS -> FADD2 -> FFMA2 -> MUFU -> FADD2 -> F2FP chains of several chunks overlap: measured
//     2400 cycles for the two groups' tiles together against the MUFU pipe's floor of 2048
//     (profiles/r02z_attention_timeline.txt, r02z_pipe_probe.txt);
//   * penalty LUT in four copies shifted by one float each and padded by 0 / 12 / 20 / 28 floats: every
//     thread reads its 128 consecutive penalties with aligned, bank-conflict-free LDS.128;
//   * P (bf16) is handed to the PV product THROUGH TENSOR MEMORY (tcgen05.st, then tcgen05.mma with the A
//     operand in TMEM): one hand-over per tile, no generic -> async proxy fence, half the shared-memory
//     traffic of the tile (61.4 -> 53.2 us together with the straight-line block);
//   * the item's output goes through a per-warp swizzled staging tile and one TMA store (a thread owns a
//     128-byte row: stored directly, every STG.128 touched 32 rows);
//   * group 1 drops a third of a tile behind group 0 once, after the first item: the two groups share one
//     MUFU pipe per scheduler and otherwise run -- and wait -- in lockstep (51.2 -> 47.1 us).
// Measured at cfg2 (L = 375, B = 64, H = 8): 47.1 us against 61.4 us; L = 1500, B = 8, H = 16: 142 us
// against 172 us (profiles/r02z_attention_ab.txt).  Development log: profiles/r02z_attention_wide.txt.
//
// One-pass softmax: the running reference m is an overflow guard only (P is bf16, l / O are fp32 -- all
// with the fp32 exponent range), raised (with a rescale of O and l) when a row's raw maximum exceeds it by
// 2^24.  The whole row is in registers before any exponential, so there is no tile restart here.
#include <math.h>
#include <stdlib.h>

#include "host_common.h"
#include "ptx.cuh"

namespace fbkst {
namespace {

constexpr int AW_BM = 128;  // queries per item
constexpr int AW_BN = 128;  // keys per tile
constexpr int AW_HD = 64;
constexpr int AW_QB = AW_BM * AW_HD * 2;  // 16 KB
constexpr int AW_KB = AW_BN * AW_HD * 2;  // 16 KB (K tile; V tile = two 8 KB halves)
// P is handed to the PV product through tensor memory (A operand of tcgen05.mma from TMEM), not through two
// swizzled shared-memory sub-tiles: no 64 KB store + 64 KB operand fetch per tile pair on the 128 B/clk
// shared-memory path, no generic -> async proxy fence (profiles/r02z_attention_wide.txt).
// Per-group shared-memory tile behind sP: the output staging rows (4 warps x 32 rows x 128 B).
constexpr int AW_PB = AW_BM * AW_HD * 2;  // 16 KB
constexpr int AW_KST = 3;  // K ring stages (4 measured the same: r02z_attention_wide.txt)
static_assert(AW_KST <= 4, "k_full / k_empty hold 4 barriers each");
constexpr int AW_THREADS = 384;
constexpr int AW_TABLE = 64;
constexpr int AW_SMEM_FIXED = 2 * AW_QB + AW_KST * AW_KB + 2 * AW_KB + 2 * AW_PB + 256 /*barriers*/ +
                              AW_TABLE * 16 /*item table*/ + 1024 /*align*/;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kGrow = 24.0f;  // log2 units by which a half's raw scores may exceed the reference

// penalty LUT (stored negated, log2 domain): entry o <-> (key - query) = o - lut_off, lut_off = nq * 128;
// copy r (0..3) holds lut[o + r] at index o, so a thread whose first index is = r (mod 4) reads copy r
// at the aligned index below it.  Copy r starts aw_lut_copy(r, n) floats into the LUT: n apart plus a pad of
// 0 / 12 / 20 / 28 floats, which puts the eight 16-byte reads of a quarter-warp (rows q .. q+7 read the
// overlapping windows lut[C-q .. C-q+3], i.e. copies 0,3,2,1,0,3,2,1 at aligned indices C, C-4 x4, C-8 x3)
// into eight different 4-bank groups: without the pads rows q+1 .. q+4 collide (n is a multiple of 32):
// 16 wavefronts per LDS.128 instead of 4 (profiles/r02z_attention_wide.txt).
__host__ __device__ inline int aw_lut_floats(int L) {
  return ((L + AW_BM - 1) / AW_BM) * AW_BM + ((L + AW_BN - 1) / AW_BN) * AW_BN;
}
__host__ __device__ inline int aw_lut_copy(int r, int n) { return r * n + (r ? 4 + 8 * r : 0); }
inline int aw_smem_bytes(int L, int log_penalty) {
  return AW_SMEM_FIXED + (log_penalty ? 4 * (4 * aw_lut_floats(L) + 32) : 0);
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// Cycles by which group 1 falls behind group 0 once, at the start of its item AW_STAGGER_ITEM: 51.2 -> 47.1 us
// at cfg2 L = 375.
constexpr int AW_STAGGER = 1200;
constexpr int AW_STAGGER_ITEM = 1;
// registers per thread after the split: 128 producer threads + 256 softmax threads <= 384 x 168 at launch
constexpr int AW_REGS_PRODUCER = 56;
constexpr int AW_REGS_SOFTMAX = 224;
static_assert(128 * AW_REGS_PRODUCER + 256 * AW_REGS_SOFTMAX <= 384 * 168, "register split");
constexpr int AW_IDLE_NS = 64;  // back-off of the idle load loop
// Every exponential runs on the MUFU pipe (16 ex2 per clock per SM = 1024 clocks for each 128 x 128 tile of
// each group).  Moving some of them to an FMA-pipe polynomial, and strictly alternating the two groups'
// exponential phases, were both measured and rejected (DESIGN.md section 4d, profiles/r02z_attention_wide.txt).
__device__ __forceinline__ void aw_exp4(float2 (&t)[4]) {
#pragma unroll
  for (int cc = 0; cc < 4; ++cc) {
    t[cc].x = ex2(t[cc].x);
    t[cc].y = ex2(t[cc].y);
  }
}
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// TMEM load without a memory clobber (it touches no memory: ordered against the barrier waits / fences /
// tcgen05.wait around it by `volatile`, against its consumers by the register outputs), so that the
// shared-memory loads and stores of neighbouring chunks may be scheduled across it
__device__ __forceinline__ void tmem_ld16v(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
// tcgen05.wait::ld that also "produces" the registers of the preceding loads: ties their first use to it
__device__ __forceinline__ void tmem_ld_wait16(uint32_t (&v)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                 "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]),
                 "+r"(v[15]));
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d));
}

// maximum of the first nv (warp-uniform) of 16 raw scores; -inf when nv <= 0
__device__ __forceinline__ float max16(const uint32_t (&a)[16], int nv) {
  if (nv >= 16) {
    float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
    for (int cc = 0; cc < 16; ++cc) m4[cc & 3] = fmaxf(m4[cc & 3], __uint_as_float(a[cc]));
    return fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
  }
  float m = -INFINITY;
#pragma unroll
  for (int cc = 0; cc < 16; ++cc)
    if (cc < nv) m = fmaxf(m, __uint_as_float(a[cc]));
  return m;
}

// 8 scores of one query row: p = 2^(s * log2e + pen - m), row sums into sm2, P packed to bf16
template <int LOGPEN>
__device__ __forceinline__ void aw_chunk(const uint32_t* __restrict__ s8, const float4* __restrict__ lp2, float2 negm2,
                                         float2 (&t)[4]) {
  const float2 l2e2 = make_float2(kLog2e, kLog2e);
  if (LOGPEN) {
    const float4 pa = lp2[0], pb = lp2[1];
    t[0] = fadd2(negm2, make_float2(pa.x, pa.y));
    t[1] = fadd2(negm2, make_float2(pa.z, pa.w));
    t[2] = fadd2(negm2, make_float2(pb.x, pb.y));
    t[3] = fadd2(negm2, make_float2(pb.z, pb.w));
  } else {
    t[0] = t[1] = t[2] = t[3] = negm2;
  }
#pragma unroll
  for (int cc = 0; cc < 4; ++cc)
    t[cc] = ffma2(make_float2(__uint_as_float(s8[2 * cc]), __uint_as_float(s8[2 * cc + 1])), l2e2, t[cc]);
}
// One 64-key half of a tile for one query row, all keys valid, straight-line (ONE basic block, no shared-memory
// stores: ptxas does not move the LUT loads of a chunk above the P stores of the previous one): 8 chunks of 8
// scores, row sums into sm2, P packed to bf16 into pk[32].
template <int LOGPEN>
__device__ __forceinline__ void aw_half(const uint32_t (&s0)[16], const uint32_t (&s1)[16], const uint32_t (&s2)[16],
                                        const uint32_t (&s3)[16], const float4* __restrict__ lp, float2 negm2,
                                        float2 (&sm2)[4], uint32_t* __restrict__ pk) {
#pragma unroll
  for (int ch = 0; ch < 8; ++ch) {
    const uint32_t* sq = (ch >> 1) == 0 ? s0 : ((ch >> 1) == 1 ? s1 : ((ch >> 1) == 2 ? s2 : s3));
    float2 t[4];
    aw_chunk<LOGPEN>(sq + (ch & 1) * 8, lp + 2 * ch, negm2, t);
    aw_exp4(t);
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
      sm2[cc] = fadd2(sm2[cc], t[cc]);
      pk[4 * ch + cc] = pack_bf16x2(t[cc].x, t[cc].y);
    }
  }
}
// Optional timeline of CTA 0 (compiled in only with -DFBKST_ATTN_TRACE, scripts/trace_attn.py): 16 x int64 per
// key tile of the CTA's stream, row = 2 * (tile count of the group) + group:  [0] S seen  [1] S in registers
// [2] guard done  [3] P computed  [4] P buffer free  [5] P handed over  [9] last PV of the item seen
// [10] item stored  [11] QK issued  [12] PV issued  [14] K load issued
__device__ long long* g_aw_trace = nullptr;
#ifdef FBKST_ATTN_TRACE
#define AW_TRACE(tile, slot)                                                        \
  do {                                                                              \
    if (trace != nullptr && (tile) < 64) trace[(tile) * 16 + (slot)] = clock64();   \
  } while (0)
#else
#define AW_TRACE(tile, slot) \
  do {                       \
  } while (0)
#endif

struct WItem {
  int w, q0, b, h, len, n_kv;  // n_kv == 0: tile of padded queries (zero fill, no pipeline work)
};
__device__ __forceinline__ int4 aw_decode(int w, const int* __restrict__ lengths, int L, int H, int nq) {
  const int qt = w % nq, bh = w / nq;
  const int b = bh / H, h = bh - b * H;
  const int q0 = qt * AW_BM;
  const int len = min(__ldg(lengths + b), L);
  return make_int4(q0, b, h, q0 < len ? len : 0);  // length 0: a tile of padded queries
}
// key tiles of an item, derived where the item is read (an 8-bit count packed beside the length wraps at 256
// tiles, L > 32640)
__device__ __forceinline__ int aw_n_kv(int len) { return static_cast<unsigned>(len + AW_BN - 1) / AW_BN; }
struct WList {
  const int4* table;  // shared memory: the CTA's first AW_TABLE items, decoded once
  const int* lengths;
  int L, H, nq, n_items;
  __device__ __forceinline__ void get(WItem& it, int k) const {
    it.w = blockIdx.x + k * gridDim.x;
    if (it.w >= n_items) return;
    const int4 r = (k < AW_TABLE) ? table[k] : aw_decode(it.w, lengths, L, H, nq);
    it.q0 = r.x;
    it.b = r.y;
    it.h = r.z;
    it.len = r.w;
    it.n_kv = aw_n_kv(it.len);
  }
};
// Tile stream of one softmax group: items k = grp, grp + 2, ... of the CTA's list, key tiles in order.
struct WCursor {
  WItem it;
  int k, j;       // index in the CTA's item list, key tile inside the item
  uint32_t c, n;  // tiles / items of this group before the current one
  __device__ __forceinline__ void seek(const WList& items) {
    for (;; k += 2) {
      items.get(it, k);
      if (it.w >= items.n_items || it.n_kv > 0) return;
    }
  }
  __device__ __forceinline__ void init(const WList& items, int grp) {
    k = grp; j = 0; c = 0; n = 0;
    seek(items);
  }
  __device__ __forceinline__ bool valid(int n_items) const { return it.w < n_items; }
  __device__ __forceinline__ void advance(const WList& items) {
    ++c;
    if (++j == it.n_kv) {
      j = 0; ++n; k += 2;
      seek(items);
    }
  }
};

template <int LOGPEN>
__global__ void __launch_bounds__(AW_THREADS, 1)
    attention_fwd_wide_kernel(const __grid_constant__ CUtensorMap tm128, const __grid_constant__ CUtensorMap tmO,
                              __nv_bfloat16* __restrict__ out, const int* __restrict__ lengths, int L, int B, int H,
                              const int* __restrict__ q_limit) {
  const int D = H * AW_HD;
  const int nq = (L + AW_BM - 1) / AW_BM;
  const int n_items = nq * B * H;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
#ifdef FBKST_ATTN_TRACE
  long long* trace = (blockIdx.x == 0 && lane == 0 && (warp < 4 || (warp & 3) == 0)) ? g_aw_trace : nullptr;
#endif
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sQ = smem;                 // 2 x 16 KB: one per group
  uint8_t* sK = sQ + 2 * AW_QB;       // AW_KST stages, shared by both groups (fixed interleaved order)
  uint8_t* sV = sK + AW_KST * AW_KB;  // one 16 KB tile (128 keys) per group
  uint8_t* sP = sV + 2 * AW_KB;       // per group: the output staging rows
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * AW_PB);
  int4* sItems = reinterpret_cast<int4*>(bars + 32);
  float* sLut = reinterpret_cast<float*>(sItems + AW_TABLE);
  uint64_t* q_full = bars + 0;    // [2]
  uint64_t* q_empty = bars + 2;   // [2]
  uint64_t* k_full = bars + 4;    // [AW_KST <= 4]
  uint64_t* k_empty = bars + 8;   // [AW_KST <= 4]
  uint64_t* v_full = bars + 12;   // [2]
  uint64_t* s_full = bars + 14;   // [2]
  uint64_t* p_full = bars + 16;   // [2]  P[g] written (128 arrivals)
  uint64_t* pv_done = bars + 18;  // [2]  the PV product of the group's tile has completed: P[g] / V[g] free, O[g] updated
  uint64_t* s_free = bars + 20;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 26);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm128);
    tma_prefetch_desc(&tmO);
    for (int s = 0; s < AW_KST; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&k_empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&q_full[s], 1);
      mbar_init(&q_empty[s], 1);
      mbar_init(&v_full[s], 1);
      mbar_init(&s_full[s], 1);
      mbar_init(&p_full[s], 128);
      mbar_init(&pv_done[s], 1);
      mbar_init(&s_free[s], 128);
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  pdl_launch_dependents();
  pdl_wait();
  if (threadIdx.x >= 128 && threadIdx.x < 128 + AW_TABLE) {
    const int w = blockIdx.x + (threadIdx.x - 128) * gridDim.x;
    if (w < n_items) sItems[threadIdx.x - 128] = aw_decode(w, lengths, L, H, nq);
  }
  const WList items{sItems, lengths, L, H, nq, n_items};
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_O = tmem_base + 2 * AW_BN;  // S[0] +0, S[1] +128, O[0] +256, O[1] +320, P[0] +384, P[1] +448
  const uint32_t tmem_P = tmem_O + 2 * AW_HD;     // P[g]: 128 bf16 keys = 64 columns per row

  // Fixed interleaved order of the two groups' tile streams on the shared K ring (identical in the load
  // warp and the QK warp): the group whose turn it is, or the other one when that stream is exhausted.
#define AW_PICK(c0, c1, turn) (((turn) == 0) ? ((c0).valid(n_items) ? 0 : 1) : ((c1).valid(n_items) ? 1 : 0))

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(AW_REGS_PRODUCER));
    if (warp == 0) {
      // ------------------------------------------------ TMA loads (Q, K, V halves): event loop over
      // non-blocking mbarrier.test_wait probes, so no load queues behind a wait that belongs to the other group
      WCursor kc0, kc1, vc0, vc1;
      kc0.init(items, 0); kc1.init(items, 1); vc0.init(items, 0); vc1.init(items, 1);
      int kturn = 0;
      uint32_t gk = 0;
      auto try_k = [&](WCursor& c, int g) -> bool {
        const uint32_t ks = gk % AW_KST;
        if (!mbar_test_wait(&k_empty[ks], ((gk / AW_KST) & 1) ^ 1)) return false;
        if (c.j == 0 && !mbar_test_wait(&q_empty[g], (c.n & 1) ^ 1)) return false;
        const int cq = c.it.h * AW_HD, ck = D + cq;
        if (elect_one()) {
          if (c.j == 0) {
            mbar_arrive_expect_tx(&q_full[g], AW_QB);
            tma_load_3d(sQ + g * AW_QB, &tm128, &q_full[g], cq, c.it.b, c.it.q0);
          }
          mbar_arrive_expect_tx(&k_full[ks], AW_KB);
          tma_load_3d(sK + ks * AW_KB, &tm128, &k_full[ks], ck, c.it.b, c.j * AW_BN);
          AW_TRACE(2 * c.c + g, 14);
        }
        __syncwarp();
        ++gk;
        c.advance(items);
        return true;
      };
      auto try_v = [&](WCursor& c, int g) -> bool {
        // V[g] was read by the PV product of the group's previous tile
        if (c.c >= 1 && !mbar_test_wait(&pv_done[g], (c.c - 1) & 1)) return false;
        const int cv = 2 * D + c.it.h * AW_HD;
        if (elect_one()) {
          mbar_arrive_expect_tx(&v_full[g], AW_KB);
          tma_load_3d(sV + g * AW_KB, &tm128, &v_full[g], cv, c.it.b, c.j * AW_BN);
        }
        __syncwarp();
        c.advance(items);
        return true;
      };
      uint32_t idle = 0;
      for (;;) {
        const bool k_left = kc0.valid(n_items) || kc1.valid(n_items);
        const bool v_left = vc0.valid(n_items) || vc1.valid(n_items);
        if (!k_left && !v_left) break;
        bool progressed = false;
        if (v_left) {
          if (vc0.valid(n_items) && try_v(vc0, 0)) progressed = true;
          if (vc1.valid(n_items) && try_v(vc1, 1)) progressed = true;
        }
        if (k_left) {
          const bool ok = (AW_PICK(kc0, kc1, kturn) == 0) ? try_k(kc0, 0) : try_k(kc1, 1);
          if (ok) { kturn ^= 1; progressed = true; }
        }
        if (!progressed) __nanosleep(AW_IDLE_NS);
#if FBKST_WATCHDOG
        idle = progressed ? 0 : idle + 1;
        if (idle > (1u << 26)) {
          printf("fbkst: wide attention load loop watchdog block=%d\n", blockIdx.x);
          __trap();
        }
#endif
      }
    } else if (warp == 1) {
      // ------------------------------------------------ QK issuer (blocking, in the K ring's order)
      constexpr uint32_t IDESC_QK = idesc_bf16_f32(AW_BM, AW_BN, 0, 0);
      WCursor qc0, qc1;
      qc0.init(items, 0); qc1.init(items, 1);
      int qturn = 0;
      uint32_t gq = 0;
      auto issue_qk = [&](WCursor& c, int g) {
        // S[g] must have been pulled into registers by the group's previous tile
        if (c.c >= 1) mbar_wait(&s_free[g], (c.c - 1) & 1);
        if (c.j == 0) mbar_wait(&q_full[g], c.n & 1);
        const uint32_t ks = gq % AW_KST;
        mbar_wait(&k_full[ks], (gq / AW_KST) & 1);
        tc_fence_after();
        const uint64_t qdesc = desc_kmajor_sw128(smem_u32(sQ + g * AW_QB));
        const uint64_t kdesc = desc_kmajor_sw128(smem_u32(sK + ks * AW_KB));
        const uint32_t d_tmem = tmem_base + g * AW_BN;
        const bool last = c.j + 1 == c.it.n_kv;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < AW_HD / 16; ++k) umma_bf16_ss(d_tmem, qdesc + 2 * k, kdesc + 2 * k, IDESC_QK, k != 0);
          umma_commit(&s_full[g]);
          umma_commit(&k_empty[ks]);
          if (last) umma_commit(&q_empty[g]);  // Q[g] may be overwritten once these MMAs have completed
          AW_TRACE(2 * c.c + g, 11);
        }
        __syncwarp();
        ++gq;
        c.advance(items);
      };
      while (qc0.valid(n_items) || qc1.valid(n_items)) {
        if (AW_PICK(qc0, qc1, qturn) == 0) issue_qk(qc0, 0); else issue_qk(qc1, 1);
        qturn ^= 1;
      }
    } else {
      // ------------------------------------------------ PV issuer of group (warp - 2): blocking, own stream
      constexpr uint32_t IDESC_PV = idesc_bf16_f32(AW_BM, AW_HD, 0, 1);
      const int g = warp - 2;
      WCursor pc;
      pc.init(items, g);
      const uint32_t va = smem_u32(sV + g * AW_KB);
      while (pc.valid(n_items)) {
        const uint32_t ph = pc.c & 1;
        mbar_wait(&p_full[g], ph);
        mbar_wait(&v_full[g], ph);
        tc_fence_after();
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < 8; ++kk) {
            // A = P[g] from tensor memory: 128 lanes (query rows) x 8 columns (16 bf16 keys) per k-step
            umma_bf16_ts(tmem_O + g * AW_HD, tmem_P + g * (AW_BN / 2) + 8 * kk,
                         desc_mnmajor_sw128(va + kk * 2048, AW_KB), IDESC_PV, (pc.j > 0) || kk != 0);
          }
          umma_commit(&pv_done[g]);
          AW_TRACE(2 * pc.c + g, 12);
        }
        __syncwarp();
        pc.advance(items);
      }
    }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(AW_REGS_SOFTMAX));
    // ---- softmax / correction / output: thread <-> (query row of the group's own item)
    const int grp = (warp - 4) >> 2;
    const int q = (warp & 3) * 32 + lane;  // row in the tile == TMEM lane
    const int st = threadIdx.x - 128;      // 0..255
    const uint32_t lane_addr = static_cast<uint32_t>((warp & 3) * 32) << 16;
    const uint32_t tS = tmem_base + lane_addr + grp * AW_BN;
    const uint32_t tO = tmem_O + lane_addr + grp * AW_HD;
    const uint32_t tP = tmem_P + lane_addr + grp * (AW_BN / 2);
    uint64_t* my_s_full = &s_full[grp];
    uint64_t* my_p_full = &p_full[grp];
    uint64_t* my_pv_done = &pv_done[grp];
    uint64_t* my_s_free = &s_free[grp];
    uint8_t* stage_warp = sP + grp * AW_PB + (warp & 3) * 4096;  // epilogue staging: 32 rows x 128 B
    const int lut_off = nq * AW_BM;
    const int lut_n = aw_lut_floats(L);
    if (LOGPEN) {
      for (int o = st; o < 4 * lut_n; o += 256) {
        const int r = o / lut_n, oo = o - r * lut_n;
        const int d = abs(oo + r - lut_off);
        sLut[aw_lut_copy(r, lut_n) + oo] = (d > 1) ? -__log2f((float)d) : 0.0f;
      }
      named_bar_sync(1, 256);
    }
    // first LUT index of row i for key k0 is lut_off - i + k0 = r (mod 4) with r = (-q) & 3
    const int lut_r = (4 - (q & 3)) & 3;
    uint32_t c = 0;  // key tiles of this group before the current one
    const int q_lim = q_limit ? __ldg(q_limit) : L;  // (after pdl_wait: written by the previous kernel)
    WItem it;
    // (item index, stride and count pinned in registers: ptxas otherwise rebuilds them from the kernel
    // parameters and special registers at every item, ~8 % of the softmax warps' time in the first profile)
    // The NEXT item of the group is decoded while the current one is processed (its table entry, the
    // special registers and kernel parameters behind the index arithmetic are long-latency reads that
    // otherwise sit between two items: ~8 % of the softmax warps' samples in the first profile).
    int w_cur = blockIdx.x + grp * gridDim.x;
    int4 r_cur = make_int4(0, 0, 0, 0);
    if (w_cur < n_items) r_cur = (grp < AW_TABLE) ? sItems[grp] : aw_decode(w_cur, lengths, L, H, nq);
    for (int k = grp; w_cur < n_items; k += 2) {
      it.w = w_cur;
      it.q0 = r_cur.x;
      it.b = r_cur.y;
      it.h = r_cur.z;
      it.len = r_cur.w;
      it.n_kv = aw_n_kv(it.len);
      w_cur += 2 * gridDim.x;
      if (w_cur < n_items) r_cur = (k + 2 < AW_TABLE) ? sItems[k + 2] : aw_decode(w_cur, lengths, L, H, nq);
      const int i = it.q0 + q;
      __nv_bfloat16* orow = out + ((size_t)i * B + it.b) * D + it.h * AW_HD;
      if (it.n_kv == 0) {  // tile of padded queries: defined (finite) output, no pipeline work
        if (i < L && it.q0 < q_lim) {  // tiles at or beyond the caller's row limit are never read: skip
          uint4* op = reinterpret_cast<uint4*>(orow);
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) op[jj] = make_uint4(0, 0, 0, 0);
        }
        continue;
      }
      const float4* lut_row = reinterpret_cast<const float4*>(sLut + aw_lut_copy(lut_r, lut_n) + (lut_off - i - lut_r));
      float m_used = -INFINITY, l = 0.0f;
      for (int j = 0; j < it.n_kv; ++j, ++c) {
        const uint32_t ph = c & 1;
        const int k0 = j * AW_BN;
        const int nvalid = min(AW_BN, it.len - k0);
        const float4* lp = lut_row + (k0 >> 2);
        float2 sm2[4];
        uint32_t s[8][16], pk[64];
        // The two groups share one MUFU pipe per scheduler.  Started together they stay in lockstep: both run
        // their exponentials at the same time (2400 cycles for the pair, the pipe's floor being 2048) and both
        // sit in their guard / hand-over / TMEM-load phases at the same time (~1100 cycles per tile in which
        // the pipe idles: timeline in profiles/r02z_attention_wide.txt).  Group 1 therefore drops a third of a
        // tile behind, once, after the instruction-cache-cold first item (which re-aligns the groups)
        if (grp == 1 && j == 0 && k == 1 + 2 * AW_STAGGER_ITEM) {
          const long long t_go = clock64() + AW_STAGGER;
          while (clock64() < t_go) {
          }
        }
        mbar_wait(my_s_full, ph);
        AW_TRACE(2 * c + grp, 0);
        tc_fence_after();
        // the whole 128-score row goes to registers and S[grp] is handed back at once: the QK product of the
        // group's next tile runs under this tile's exponentials
#pragma unroll
        for (int a = 0; a < 8; ++a) tmem_ld16v(tS + 16 * a, s[a]);
#pragma unroll
        for (int a = 0; a < 4; ++a) sm2[a] = make_float2(0.f, 0.f);
#pragma unroll
        for (int a = 0; a < 8; ++a) tmem_ld_wait16(s[a]);
        AW_TRACE(2 * c + grp, 1);
        tc_fence_before();
        mbar_arrive(my_s_free);
        if (nvalid != AW_BN) {
          // last tile of the utterance: scores of keys at or beyond the length become -inf in the registers
          // (warp-uniform per 16-score group: untouched / 16 selects / 16 moves), so that the guard and the
          // exponentials below have ONE straight-line form for every tile
#pragma unroll
          for (int a = 0; a < 8; ++a) {
            const int nv = nvalid - 16 * a;
            if (nv < 16) {
#pragma unroll
              for (int cc = 0; cc < 16; ++cc)
                if (cc >= nv) s[a][cc] = 0xff800000u;
            }
          }
        }
        {
          float mx = -INFINITY;
#pragma unroll
          for (int a = 0; a < 8; ++a) mx = fmaxf(mx, max16(s[a], 16));
          const float m_row = mx * kLog2e;
          const bool grow = m_row > m_used + kGrow;
          if (__any_sync(0xffffffffu, grow)) {
            const float m_next = grow ? m_row : m_used;
            if (j > 0) {
              mbar_wait(my_pv_done, ph ^ 1);  // O[grp] quiescent: the PV product of the previous tile has completed
              const float alpha = ex2(m_used - m_next);
              tc_fence_after();
              // rare path: rolled, 8 columns at a time
#pragma unroll 1
              for (int cb = 0; cb < AW_HD; cb += 8) {
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
        const float2 negm2 = make_float2(-m_used, -m_used);
        AW_TRACE(2 * c + grp, 2);
        // all 16 chunks of 8 scores in ONE basic block, P packed into registers (they replace the score
        // registers as those die) ...
        aw_half<LOGPEN>(s[0], s[1], s[2], s[3], lp, negm2, sm2, pk);
        aw_half<LOGPEN>(s[4], s[5], s[6], s[7], lp + 16, negm2, sm2, pk + 32);
        AW_TRACE(2 * c + grp, 3);
        // ... and stored once the PV product of the previous tile, which read this buffer, has completed
        if (c >= 1) mbar_wait(my_pv_done, ph ^ 1);
        AW_TRACE(2 * c + grp, 4);
        tc_fence_after();
        tmem_st32(tP, *reinterpret_cast<uint32_t(*)[32]>(&pk[0]));
        tmem_st32(tP + 32, *reinterpret_cast<uint32_t(*)[32]>(&pk[32]));
        l += (sm2[0].x + sm2[0].y) + (sm2[1].x + sm2[1].y) + (sm2[2].x + sm2[2].y) + (sm2[3].x + sm2[3].y);
        tmem_st_wait();
        tc_fence_before();  // (also orders the O reads of the previous item's epilogue / a rescale before PV)
        mbar_arrive(my_p_full);
        AW_TRACE(2 * c + grp, 5);
      }
      // ---- item epilogue (this group only): O / l -> bf16.  A thread owns a query row (128 B); stored
      // straight from there every STG.128 touches 32 rows (32 sectors per instruction: 2250 cycles per item
      // in the first timeline, and the next item's shared-memory loads queued behind them).  Each warp stages
      // its 32 rows (4 KB, 128B-swizzled) in shared memory and ONE lane hands them to the TMA unit as a
      // {64 columns, 1 utterance, 32 rows} box of the [L, B, D] output (rows at or beyond L are clipped).
      mbar_wait(my_pv_done, (c - 1) & 1);  // O[grp] final
      AW_TRACE(2 * (c - 1) + grp, 9);
      tc_fence_after();
      const float inv = 1.0f / l;
      {
        uint32_t o0[32], o1[32];
        tmem_ld32(tO, o0);
        tmem_ld32(tO + 32, o1);
        // the staging rows are free once the previous item's store has read them
        if (lane == 0) tma_store_wait_read<0>();
        __syncwarp();
        tmem_ld_wait();
        const uint32_t my_row = smem_u32(stage_warp) + (uint32_t)lane * 128u;
#pragma unroll
        for (int gq4 = 0; gq4 < 8; ++gq4) {
          const uint32_t* ov = (gq4 < 4) ? &o0[gq4 * 8] : &o1[(gq4 - 4) * 8];
          sts128(my_row + (((uint32_t)gq4 ^ (uint32_t)(lane & 7)) << 4),
                 pack_bf16x2(__uint_as_float(ov[0]) * inv, __uint_as_float(ov[1]) * inv),
                 pack_bf16x2(__uint_as_float(ov[2]) * inv, __uint_as_float(ov[3]) * inv),
                 pack_bf16x2(__uint_as_float(ov[4]) * inv, __uint_as_float(ov[5]) * inv),
                 pack_bf16x2(__uint_as_float(ov[6]) * inv, __uint_as_float(ov[7]) * inv));
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(&tmO, stage_warp, it.h * AW_HD, it.b, it.q0 + (warp & 3) * 32);
          tma_store_commit();
        }
      }
      // O[grp] is overwritten by the PV of the group's next tile, which waits for this group's next
      // p_full arrival (ordered after the TMEM reads above by the fence before that arrive)
      AW_TRACE(2 * (c - 1) + grp, 10);
    }
    if (lane == 0) tma_store_wait<0>();  // output stores complete (and staging rows read) before the CTA retires
  }
#undef AW_PICK
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

}  // namespace fbkst
// debug hook (not part of the public ABI): buffer of 64*16 int64, or NULL to disable
extern "C" int fbkst_debug_set_attention_wide_trace(long long* buf) {
  cudaError_t e = cudaMemcpyToSymbol(fbkst::g_aw_trace, &buf, sizeof(buf));
  return e == cudaSuccess ? 0 : -2;
}
namespace fbkst {

// Returns FBKST_OK after launching, or 1 when this shape is not served by the wide kernel (the caller
// falls through to the split-KV kernel of attention_tcgen05.cu).
int attention_wide_launch(const void* qkv, void* out, const int32_t* lengths, int L, int B, int H, int log_penalty,
                          const int32_t* q_limit, cudaStream_t st) {
  const int smem = aw_smem_bytes(L, log_penalty);
  if (smem > 227 * 1024) return 1;
  const int D = H * AW_HD;
  CUtensorMap tm128;
  uint64_t dims[3] = {(uint64_t)3 * D, (uint64_t)B, (uint64_t)L};
  uint64_t strides[2] = {(uint64_t)3 * D * 2, (uint64_t)B * 3 * D * 2};
  uint32_t box128[3] = {AW_HD, 1, 128};
  int rc = make_tensor_map(&tm128, qkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 3, dims, strides, box128, nullptr);
  if (rc) return rc;
  CUtensorMap tmO;
  {
    uint64_t odims[3] = {(uint64_t)D, (uint64_t)B, (uint64_t)L};
    uint64_t ostrides[2] = {(uint64_t)D * 2, (uint64_t)B * D * 2};
    uint32_t obox[3] = {AW_HD, 1, 32};
    rc = make_tensor_map(&tmO, out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 3, odims, ostrides, obox, nullptr);
    if (rc) return rc;
  }
  static PerDeviceFlag configured;
  if (!configured) {
    FBKST_CHECK_CUDA(cudaFuncSetAttribute(attention_fwd_wide_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          227 * 1024));
    FBKST_CHECK_CUDA(cudaFuncSetAttribute(attention_fwd_wide_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          227 * 1024));
    configured = true;
  }
  const long long n_items = (long long)((L + AW_BM - 1) / AW_BM) * B * H;
  FBKST_REQUIRE(n_items < (1ll << 30), "fbkst_attention_fwd: too many work items");
  int grid = num_sms();
  if (2 * (long long)grid > n_items) grid = (int)((n_items + 1) / 2);
  if (log_penalty)
    FBKST_CHECK_CUDA(launch_pdl(attention_fwd_wide_kernel<1>, dim3(grid), dim3(AW_THREADS), smem, st, tm128, tmO,
                                (__nv_bfloat16*)out, lengths, L, B, H, q_limit));
  else
    FBKST_CHECK_CUDA(launch_pdl(attention_fwd_wide_kernel<0>, dim3(grid), dim3(AW_THREADS), smem, st, tm128, tmO,
                                (__nv_bfloat16*)out, lengths, L, B, H, q_limit));
  return FBKST_OK;
}

}  // namespace fbkst
