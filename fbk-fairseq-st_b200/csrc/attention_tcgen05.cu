// Fused self-attention core for the ST encoder (reference: local_attention.py:115-139 with
// LogPenalty conv_transformer_layer.py:22-27): flash-style streaming softmax on tcgen05.  It serves the
// lengths the wide kernel (attention_wide.cu) cannot fit: the log penalty at L > 2560, up to L = 17216.
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
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ float lds32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Every exponential runs on the MUFU pipe: 16 ex2 per clock and SM, i.e. 512 clocks for a 128x64 tile
// whose two UMMAs need 256.  Moving part of each row to an FMA-pipe polynomial 2^x (Cody-Waite + degree-3
// minimax) was MEASURED slower (profiles/r01f_attention_poly_ab.txt, cfg2 L=375: 61.4 / 63.5 / 65.5 /
// 67.6 us for 0..3 of every 4 register pairs): the softmax warps are bound by issue slots and the MMA
// round trip, not by the MUFU pipe.

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

__global__ void __launch_bounds__(AT_THREADS, 2)
    attention_fwd_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                         __nv_bfloat16* __restrict__ out, const int* __restrict__ lengths, int L, int B,
                         int H, const int* __restrict__ q_limit) {
  const int D = H * AT_HD;
  const int nq = (L + AT_BM - 1) / AT_BM;
  const int n_items = nq * B * H;
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;

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
          tc_fence_after();
          issue_qk();
        }
        mbar_wait(&p_full[pb], ph);  // P[pb] in smem, O[pb] rescaled / read out
        mbar_wait(&v_full[pb], ph);
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
    const int n_lut = lut_off + ((L + AT_BN - 1) / AT_BN) * AT_BN;
    for (int o = st; o < n_lut; o += 256) {
      const int d = abs(o - lut_off);
      sLut[o] = (d > 1) ? -__log2f((float)d) : 0.0f;
    }
    named_bar_sync(1, 256);
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
        if (gg >= 2) mbar_wait(my_pv_done, ph ^ 1);
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
#pragma unroll
          for (int c = 0; c < 8; ++c) pn[c] = lds32(lut_addr + c * 4);
          tmem_ld_wait();
#pragma unroll
          for (int ch = 0; ch < 8; ++ch) {  // 8 columns at a time: registers, not ILP, are scarce
            uint32_t(&s0)[16] = (ch & 2) ? sb : sa;
            const int o = (ch & 1) * 8;
            float2 t[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const float2 add = fadd2(negm2, make_float2(pn[2 * c], pn[2 * c + 1]));
              t[c] = ffma2(make_float2(__uint_as_float(s0[o + 2 * c]), __uint_as_float(s0[o + 2 * c + 1])),
                           l2e2, add);
            }
            if (ch == 1 || ch == 3) tmem_ld16(tS + (ch + 3) * 8, s0);  // columns 32.. / 48.. into the freed buffer
            if (ch < 7) {  // penalties of the next 8 columns fly under the exps
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
              t[c].x = ex2(t[c].x);
              t[c].y = ex2(t[c].y);
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
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

// attention_wide.cu: one CTA per SM, 128-key tiles; returns 1 when the shape is not served
int attention_wide_launch(const void* qkv, void* out, const int32_t* lengths, int L, int B, int H, int log_penalty,
                          const int32_t* q_limit, cudaStream_t st);

}  // namespace fbkst

using namespace fbkst;

static int attention_entry(const void* qkv, void* out, const int32_t* lengths, int L, int B, int H,
                           int log_penalty, const int32_t* q_limit, fbkst_stream_t stream) {
  FBKST_REQUIRE(qkv && out && lengths, "fbkst_attention_fwd: null pointer");
  FBKST_REQUIRE(L > 0 && B > 0 && H > 0, "fbkst_attention_fwd: bad shape L=%d B=%d H=%d", L, B, H);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // wide kernel (attention_wide.cu: one CTA per SM, 128-key tiles, P through tensor memory) whenever its shared
  // memory fits: always without the penalty (no LUT), L <= 2560 with it
  int rc = attention_wide_launch(qkv, out, lengths, L, B, H, log_penalty, q_limit, st);
  if (rc != 1) return rc;
  // longer L with the penalty: the split-KV kernel above (one LUT copy: up to L = 17216)
  FBKST_REQUIRE(log_penalty, "fbkst_attention_fwd: the wide kernel declined L=%d without the penalty", L);
  const int D = H * AT_HD;
  CUtensorMap tmQ, tmKV;
  uint64_t dims[3] = {(uint64_t)3 * D, (uint64_t)B, (uint64_t)L};
  uint64_t strides[2] = {(uint64_t)3 * D * 2, (uint64_t)B * 3 * D * 2};
  uint32_t boxq[3] = {AT_HD, 1, AT_BM};
  uint32_t boxk[3] = {AT_HD, 1, AT_BN};
  rc = make_tensor_map(&tmQ, qkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 3, dims, strides, boxq, nullptr);
  if (rc) return rc;
  rc = make_tensor_map(&tmKV, qkv, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, 3, dims, strides, boxk, nullptr);
  if (rc) return rc;
  static PerDeviceFlag configured;
  if (!configured) {
    FBKST_CHECK_CUDA(cudaFuncSetAttribute(attention_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          227 * 1024));
    configured = true;
  }
  const int smem = attention_smem_bytes(L);
  FBKST_REQUIRE(smem <= 227 * 1024, "fbkst_attention_fwd: L=%d needs %d B of shared memory", L, smem);
  // persistent grid: as many CTAs as fit (2 per SM up to L ~ 3000), never more than work items
  const int per_sm = (2 * (smem + 1024) <= 228 * 1024) ? 2 : 1;
  const long long n_items = (long long)((L + AT_BM - 1) / AT_BM) * B * H;
  FBKST_REQUIRE(n_items < (1ll << 31), "fbkst_attention_fwd: too many work items");
  int grid = num_sms() * per_sm;
  if (grid > n_items) grid = (int)n_items;
  FBKST_CHECK_CUDA(launch_pdl(attention_fwd_kernel, dim3(grid), dim3(AT_THREADS), smem, st, tmQ, tmKV,
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
