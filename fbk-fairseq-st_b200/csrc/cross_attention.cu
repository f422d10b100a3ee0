// Next row N4 (SURVEY 8f): the decoder's encoder-decoder attention over the (CTC-compressed, ragged)
// encoder output during incremental generation -- reference: fairseq/modules/multihead_attention.py
// :108-367 on its static_kv path, called from fairseq/modules/transformer_layer.py:339-348, with the
// K/V cache replicated x beam by reorder_encoder_out (conv_transformer.py:315-345,
// sequence_generator.py:193-198) and re-gathered by reorder_incremental_state (:407-420).
//
// Here K and V are projected ONCE per utterance (not per beam hypothesis) into one time-major
// buffer kv [S, U, 2D]; every hypothesis row carries an index into it (row_map), so beam
// replication and beam reordering are a gather of B*beam int32 values instead of copies of
// B*beam*H*S*64 elements per layer.  The kernel is HBM/L2-bound byte work (q.K^T and p.V for ONE
// query per row: 4 flop per K/V byte): no tensor cores, 16-byte loads, fp32 softmax.
//
//   CTA  = (utterance u, head h): it collects the hypothesis rows b with row_map[b] == u and serves
//          ALL of them (x tgt_len queries each) from one pass over K_h and V_h of the utterance, in
//          chunks of 8 query rows: the K/V bytes are read once per chunk instead of once per row
//          (beam 5 -> 5x less L2 traffic than a CTA per row, and U*H CTAs fill the 148 SMs).
//   scores  lane <-> key: a lane pulls a whole K row (bf16: 128 bytes, 8 x LDG.128; fp32: 256 bytes,
//           16 x LDG.128) into registers as 64 floats and dots it with the (up to) 8 queries of the
//           chunk, broadcast from shared memory
//   softmax fp32, warp <-> query row, probabilities stay in shared memory ([S][8] floats)
//   p.V     lane <-> two output dims, the 8 warps split the keys (a warp reads one coalesced V row
//           per key), partial sums reduced through shared memory in a fixed order
//   weights per head straight from shared memory; the head average the reference returns
//           (multihead_attention.py:355-362) is a second tiny kernel over the per-head buffer, so the
//           summation order over heads is fixed (no atomics).
//
// One kernel body serves both operand types (template on the element type T): bf16 q / kv / out
// (fbkst_xattn_fwd) and fp32 (fbkst_xattn_fwd_f32, the fp32-accurate decode path).  Only the loads
// and stores differ; arithmetic and summation order are the same fp32 FMAs for both.
#include <math.h>

#include <cuda_bf16.h>

#include "host_common.h"

namespace fbkst {

constexpr int XA_HD = 64;
constexpr int XA_RC = 8;       // query rows served per pass over K/V
constexpr int XA_WARPS = 8;
constexpr int XA_THREADS = XA_WARPS * 32;
constexpr int XA_SCAN = 1024;  // hypothesis rows scanned per list refill

__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

// two consecutive elements (8-byte aligned for fp32, 4-byte for bf16) as floats
__device__ __forceinline__ float2 xa_ld2(const __nv_bfloat16* p) {
  const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(p));
  return make_float2(bf16_lo(w), bf16_hi(w));
}
__device__ __forceinline__ float2 xa_ld2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }

__device__ __forceinline__ void xa_st2(__nv_bfloat16* p, float2 v) {
  *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(v.x, v.y);
}
__device__ __forceinline__ void xa_st2(float* p, float2 v) { *reinterpret_cast<float2*>(p) = v; }

// one 64-element head row (16-byte aligned) -> kf[64]
__device__ __forceinline__ void xa_ld_row(const __nv_bfloat16* p, float (&kf)[XA_HD]) {
  const uint4* kp = reinterpret_cast<const uint4*>(p);
  uint4 kr[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) kr[i] = __ldg(kp + i);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    kf[8 * i + 0] = bf16_lo(kr[i].x); kf[8 * i + 1] = bf16_hi(kr[i].x);
    kf[8 * i + 2] = bf16_lo(kr[i].y); kf[8 * i + 3] = bf16_hi(kr[i].y);
    kf[8 * i + 4] = bf16_lo(kr[i].z); kf[8 * i + 5] = bf16_hi(kr[i].z);
    kf[8 * i + 6] = bf16_lo(kr[i].w); kf[8 * i + 7] = bf16_hi(kr[i].w);
  }
}
__device__ __forceinline__ void xa_ld_row(const float* p, float (&kf)[XA_HD]) {
  const float4* kp = reinterpret_cast<const float4*>(p);
#pragma unroll
  for (int i = 0; i < XA_HD / 4; ++i) {
    const float4 v = __ldg(kp + i);
    kf[4 * i + 0] = v.x; kf[4 * i + 1] = v.y; kf[4 * i + 2] = v.z; kf[4 * i + 3] = v.w;
  }
}

static inline size_t xattn_smem_bytes(int S) {
  return sizeof(int) * (XA_SCAN + 4) + sizeof(float) * (XA_RC * XA_HD + XA_WARPS * XA_RC * XA_HD + XA_RC) +
         sizeof(float) * (size_t)S * XA_RC;
}

// A hypothesis row whose map entry is outside [0, U) belongs to no CTA: the CTAs of utterance 0 give
// it defined zeros (rare path, kept out of line).
template <typename T>
__device__ __noinline__ void xattn_zero_row(T* out, float* attn_w, int b, int h, int S, int bsz, int tgt_len,
                                            int D) {
  for (int t = 0; t < tgt_len; ++t) {
    uint4* o = reinterpret_cast<uint4*>(out + ((size_t)t * bsz + b) * D + h * XA_HD);
    for (int c = 0; c < XA_HD * (int)sizeof(T) / 16; ++c) o[c] = make_uint4(0u, 0u, 0u, 0u);
    if (attn_w != nullptr) {
      float* w = attn_w + (((size_t)h * bsz + b) * tgt_len + t) * S;
      for (int k = 0; k < S; ++k) w[k] = 0.0f;
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(XA_THREADS)
    xattn_fwd_kernel(const T* __restrict__ q, const T* __restrict__ kv, const uint8_t* __restrict__ mask,
                     const int* __restrict__ row_map, T* __restrict__ out, float* __restrict__ attn_w, int S,
                     int U, int bsz, int tgt_len, int H) {
  extern __shared__ __align__(16) uint8_t xa_raw[];
  int* s_list = reinterpret_cast<int*>(xa_raw);                 // [XA_SCAN] hypothesis rows of this utterance
  int* s_n = s_list + XA_SCAN;                                  // [4]
  float* s_q = reinterpret_cast<float*>(s_n + 4);               // [RC][64]
  float* s_red = s_q + XA_RC * XA_HD;                           // [WARPS][RC][64]
  float* s_inv = s_red + XA_WARPS * XA_RC * XA_HD;              // [RC]
  float* s_p = s_inv + XA_RC;                                   // [S][RC] scores -> probabilities
  const int D = H * XA_HD;
  const int u = blockIdx.x / H, h = blockIdx.x - u * H;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const size_t row_stride = (size_t)U * 2 * D;  // elements between consecutive keys
  const T* kbase = kv + (size_t)u * 2 * D + h * XA_HD;
  const uint8_t* mrow = mask ? mask + (size_t)u * S : nullptr;

  // Pull this CTA's K_h and V_h rows (128 or 256 bytes per key each) towards L2 now: they do not
  // depend on the row list, and every later phase is a chain of dependent round trips (scan ->
  // queries -> K -> softmax -> V) that would otherwise each pay HBM latency.
  for (int s = tid; s < S; s += XA_THREADS) {
    const T* kp = kbase + (size_t)s * row_stride;
#pragma unroll
    for (int c = 0; c < XA_HD * (int)sizeof(T); c += 128) {  // one prefetch per 128-byte line
      asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(kp) + c));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(kp + D) + c));
    }
  }
  for (int b0 = 0; b0 < bsz; b0 += XA_SCAN) {
    // ---- hypothesis rows of this utterance in [b0, b0 + XA_SCAN)
    if (tid == 0) *s_n = 0;
    __syncthreads();
    int rms[XA_SCAN / XA_THREADS];
#pragma unroll
    for (int k = 0; k < XA_SCAN / XA_THREADS; ++k) {
      const int b = b0 + k * XA_THREADS + tid;
      rms[k] = b < bsz ? __ldg(row_map + b) : -2;
    }
#pragma unroll
    for (int k = 0; k < XA_SCAN / XA_THREADS; ++k) {
      const int i = k * XA_THREADS;
      const int b = b0 + i + tid;
      const int rm = rms[k];
      const bool hit = rm == u;
      if (u == 0 && b < bsz && (rm < 0 || rm >= U)) xattn_zero_row<T>(out, attn_w, b, h, S, bsz, tgt_len, D);
      const unsigned bal = __ballot_sync(0xffffffffu, hit);
      // the order of the list is irrelevant: every row is computed independently of its chunk mates
      int base = 0;
      if (lane == 0 && bal != 0u) base = atomicAdd(s_n, __popc(bal));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (hit) s_list[base + __popc(bal & ((1u << lane) - 1))] = b;
      if (b0 + i + XA_THREADS >= bsz) break;  // block-uniform
    }
    __syncthreads();
    const int n_rows = *s_n * tgt_len;
    for (int r0 = 0; r0 < n_rows; r0 += XA_RC) {
      const int nr = min(XA_RC, n_rows - r0);
      // ---- the chunk's queries (head slice) as fp32 in shared memory; unused rows are zero
      for (int i = tid; i < XA_RC * (XA_HD / 2); i += XA_THREADS) {
        const int j = i / (XA_HD / 2), c = i - j * (XA_HD / 2);
        float2 v = make_float2(0.f, 0.f);
        if (j < nr) {
          const int idx = r0 + j;
          const int b = s_list[idx / tgt_len], t = idx % tgt_len;
          v = xa_ld2(q + ((size_t)t * bsz + b) * D + h * XA_HD + 2 * c);
        }
        reinterpret_cast<float2*>(s_q)[i] = v;
      }
      __syncthreads();
      // ---- scores: lane <-> key
      for (int s = warp * 32 + lane; s < S; s += XA_THREADS) {
        float kf[XA_HD];
        xa_ld_row(kbase + (size_t)s * row_stride, kf);
        const bool masked = mrow && mrow[s];  // multihead_attention.py:330-335
        // rolled over the rows on purpose: every CTA runs this code once, cold -- the fully unrolled
        // version (6k instructions) spent its time in instruction fetch (profiles/r01f_ncu_xattn_v2_unrolled.txt)
        float* dst = s_p + (size_t)s * XA_RC;
#pragma unroll 1
        for (int j = 0; j < nr; ++j) {
          float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
          const float4* qp = reinterpret_cast<const float4*>(s_q + j * XA_HD);
#pragma unroll
          for (int i = 0; i < XA_HD / 4; ++i) {
            const float4 qv = qp[i];  // broadcast
            a0 = fmaf(qv.x, kf[4 * i + 0], a0);
            a1 = fmaf(qv.y, kf[4 * i + 1], a1);
            a2 = fmaf(qv.z, kf[4 * i + 2], a2);
            a3 = fmaf(qv.w, kf[4 * i + 3], a3);
          }
          dst[j] = masked ? -INFINITY : (a0 + a1) + (a2 + a3);
        }
        for (int j = nr; j < XA_RC; ++j) dst[j] = 0.0f;  // unused rows: finite, never read back
      }
      __syncthreads();
      // ---- softmax (fp32, like utils.softmax on the float scores: :340-343): warp <-> row
      for (int j = warp; j < nr; j += XA_WARPS) {
        float mx = -INFINITY;
        for (int s = lane; s < S; s += 32) mx = fmaxf(mx, s_p[(size_t)s * XA_RC + j]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        float sum = 0.0f;
        if (mx > -INFINITY) {
          for (int s = lane; s < S; s += 32) {
            const float p = exp2f((s_p[(size_t)s * XA_RC + j] - mx) * 1.4426950408889634f);
            s_p[(size_t)s * XA_RC + j] = p;
            sum += p;
          }
        } else {  // every key masked (the reference would produce NaN): defined zero output
          for (int s = lane; s < S; s += 32) s_p[(size_t)s * XA_RC + j] = 0.0f;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if (lane == 0) s_inv[j] = sum > 0.0f ? 1.0f / sum : 0.0f;
      }
      __syncthreads();
      // ---- p.V: lane <-> output dims (2 * lane, 2 * lane + 1); warp w takes keys w, w + 4, ...
      {
        const T* vbase = kbase + D + 2 * lane;
        float acc[XA_RC][2];
#pragma unroll
        for (int j = 0; j < XA_RC; ++j) acc[j][0] = acc[j][1] = 0.0f;
        int s = warp;
        for (; s + 7 * XA_WARPS < S; s += 8 * XA_WARPS) {
          float2 vv[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) vv[i] = xa_ld2(vbase + (size_t)(s + i * XA_WARPS) * row_stride);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4* pp = reinterpret_cast<const float4*>(s_p + (size_t)(s + i * XA_WARPS) * XA_RC);
            const float4 p0 = pp[0], p1 = pp[1];  // broadcast
            const float v0 = vv[i].x, v1 = vv[i].y;
            acc[0][0] = fmaf(p0.x, v0, acc[0][0]); acc[0][1] = fmaf(p0.x, v1, acc[0][1]);
            acc[1][0] = fmaf(p0.y, v0, acc[1][0]); acc[1][1] = fmaf(p0.y, v1, acc[1][1]);
            acc[2][0] = fmaf(p0.z, v0, acc[2][0]); acc[2][1] = fmaf(p0.z, v1, acc[2][1]);
            acc[3][0] = fmaf(p0.w, v0, acc[3][0]); acc[3][1] = fmaf(p0.w, v1, acc[3][1]);
            acc[4][0] = fmaf(p1.x, v0, acc[4][0]); acc[4][1] = fmaf(p1.x, v1, acc[4][1]);
            acc[5][0] = fmaf(p1.y, v0, acc[5][0]); acc[5][1] = fmaf(p1.y, v1, acc[5][1]);
            acc[6][0] = fmaf(p1.z, v0, acc[6][0]); acc[6][1] = fmaf(p1.z, v1, acc[6][1]);
            acc[7][0] = fmaf(p1.w, v0, acc[7][0]); acc[7][1] = fmaf(p1.w, v1, acc[7][1]);
          }
        }
        for (; s < S; s += XA_WARPS) {
          const float2 v = xa_ld2(vbase + (size_t)s * row_stride);
          const float4* pp = reinterpret_cast<const float4*>(s_p + (size_t)s * XA_RC);
          const float4 p0 = pp[0], p1 = pp[1];
          const float v0 = v.x, v1 = v.y;
          acc[0][0] = fmaf(p0.x, v0, acc[0][0]); acc[0][1] = fmaf(p0.x, v1, acc[0][1]);
          acc[1][0] = fmaf(p0.y, v0, acc[1][0]); acc[1][1] = fmaf(p0.y, v1, acc[1][1]);
          acc[2][0] = fmaf(p0.z, v0, acc[2][0]); acc[2][1] = fmaf(p0.z, v1, acc[2][1]);
          acc[3][0] = fmaf(p0.w, v0, acc[3][0]); acc[3][1] = fmaf(p0.w, v1, acc[3][1]);
          acc[4][0] = fmaf(p1.x, v0, acc[4][0]); acc[4][1] = fmaf(p1.x, v1, acc[4][1]);
          acc[5][0] = fmaf(p1.y, v0, acc[5][0]); acc[5][1] = fmaf(p1.y, v1, acc[5][1]);
          acc[6][0] = fmaf(p1.z, v0, acc[6][0]); acc[6][1] = fmaf(p1.z, v1, acc[6][1]);
          acc[7][0] = fmaf(p1.w, v0, acc[7][0]); acc[7][1] = fmaf(p1.w, v1, acc[7][1]);
        }
#pragma unroll
        for (int j = 0; j < XA_RC; ++j)
          reinterpret_cast<float2*>(s_red + (warp * XA_RC + j) * XA_HD)[lane] = make_float2(acc[j][0], acc[j][1]);
      }
      __syncthreads();
      // ---- outputs: fixed-order sum over the warps, 1 / row sum, stored as T
      for (int i = tid; i < nr * (XA_HD / 2); i += XA_THREADS) {
        const int j = i / (XA_HD / 2), c = i - j * (XA_HD / 2);
        float2 a = make_float2(0.f, 0.f);
#pragma unroll
        for (int w = 0; w < XA_WARPS; ++w) {
          const float2 v = reinterpret_cast<const float2*>(s_red + (w * XA_RC + j) * XA_HD)[c];
          a.x += v.x;
          a.y += v.y;
        }
        const float inv = s_inv[j];
        const int idx = r0 + j;
        const int b = s_list[idx / tgt_len], t = idx % tgt_len;
        xa_st2(out + ((size_t)t * bsz + b) * D + h * XA_HD + 2 * c, make_float2(a.x * inv, a.y * inv));
      }
      if (attn_w != nullptr) {  // per-head weights [H, bsz, tgt_len, S]
        for (int j = 0; j < nr; ++j) {
          const int idx = r0 + j;
          const int b = s_list[idx / tgt_len], t = idx % tgt_len;
          float* w = attn_w + (((size_t)h * bsz + b) * tgt_len + t) * S;
          const float inv = s_inv[j];
          for (int s = tid; s < S; s += XA_THREADS) w[s] = s_p[(size_t)s * XA_RC + j] * inv;
        }
      }
      __syncthreads();
    }
  }
}

// mean over heads in a fixed order: per_head [H, n] -> avg [n]   (multihead_attention.py:360-362)
__global__ void xattn_head_mean_kernel(const float* __restrict__ per_head, float* __restrict__ avg, size_t n,
                                       int H) {
  const float invH = 1.0f / (float)H;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float a = 0.0f;
    for (int h = 0; h < H; ++h) a += per_head[(size_t)h * n + i];
    avg[i] = a * invH;
  }
}

// The launch behind both entry points: T is the element type of q, kv and out.
template <typename T>
int xattn_launch(const char* name, const void* q, const void* kv, const uint8_t* key_padding_mask,
                 const int32_t* row_map, void* out, float* attn_w, float* head_ws, int w_mode, int S, int U,
                 int bsz, int tgt_len, int H, fbkst_stream_t stream) {
  FBKST_REQUIRE(q && kv && row_map && out, "%s: null pointer", name);
  FBKST_REQUIRE(S >= 1 && U >= 1 && bsz >= 1 && tgt_len >= 1, "%s: empty problem (S=%d U=%d bsz=%d tgt_len=%d)",
                name, S, U, bsz, tgt_len);
  FBKST_REQUIRE(H >= 1 && H <= 16, "%s: heads must be in [1,16] (head_dim is 64), got %d", name, H);
  FBKST_REQUIRE(w_mode >= 0 && w_mode <= 2 && (w_mode == 0 || attn_w), "%s: bad attention-weight mode", name);
  FBKST_REQUIRE(w_mode != 1 || head_ws, "%s: head-averaged weights need the [H, bsz, tgt_len, S] workspace", name);
  FBKST_REQUIRE((reinterpret_cast<uintptr_t>(q) & (2 * sizeof(T) - 1)) == 0 &&
                    (reinterpret_cast<uintptr_t>(kv) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                "%s: q must be aligned to two elements, kv and out to 16 bytes", name);
  const size_t smem = xattn_smem_bytes(S);
  FBKST_REQUIRE(smem <= 200 * 1024, "%s: src_len %d too long (scores of 8 rows must fit in shared memory)", name, S);
  static PerDeviceFlag configured;  // one per instantiation
  if (smem > 48 * 1024 && !configured) {
    FBKST_CHECK_CUDA(
        cudaFuncSetAttribute(xattn_fwd_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    configured = true;
  }
  const long long rows = (long long)bsz * tgt_len, ctas = (long long)U * H;
  FBKST_REQUIRE(rows <= 0x7fffffffLL && ctas <= 0x7fffffffLL, "%s: problem too large", name);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* per_head = w_mode == 2 ? attn_w : (w_mode == 1 ? head_ws : nullptr);
  xattn_fwd_kernel<T><<<(unsigned)ctas, XA_THREADS, smem, st>>>(static_cast<const T*>(q), static_cast<const T*>(kv),
                                                                key_padding_mask, row_map, static_cast<T*>(out),
                                                                per_head, S, U, bsz, tgt_len, H);
  if (w_mode == 1) {
    const size_t n = (size_t)rows * S;
    const unsigned grid = (unsigned)((n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184);
    xattn_head_mean_kernel<<<grid, 256, 0, st>>>(head_ws, attn_w, n, H);
  }
  FBKST_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace fbkst

extern "C" int fbkst_xattn_fwd(const void* q, const void* kv, const uint8_t* key_padding_mask,
                               const int32_t* row_map, void* out, float* attn_w, float* head_ws, int w_mode,
                               int S, int U, int bsz, int tgt_len, int H, fbkst_stream_t stream) {
  return fbkst::xattn_launch<__nv_bfloat16>("xattn_fwd", q, kv, key_padding_mask, row_map, out, attn_w, head_ws,
                                            w_mode, S, U, bsz, tgt_len, H, stream);
}

extern "C" int fbkst_xattn_fwd_f32(const float* q, const float* kv, const uint8_t* key_padding_mask,
                                   const int32_t* row_map, float* out, float* attn_w, float* head_ws, int w_mode,
                                   int S, int U, int bsz, int tgt_len, int H, fbkst_stream_t stream) {
  return fbkst::xattn_launch<float>("xattn_fwd_f32", q, kv, key_padding_mask, row_map, out, attn_w, head_ws,
                                    w_mode, S, U, bsz, tgt_len, H, stream);
}
