// Next row N5: the decoder's self-attention during incremental generation -- reference:
// fairseq/modules/multihead_attention.py:108-367 with self_attention=True as TransformerDecoderLayer.forward calls it
// (fairseq/modules/transformer_layer.py), whose incremental path appends the step's key and value
// to the cached (bsz*beam, H, t, 64) tensors with torch.cat and gathers the whole cache again in
// reorder_incremental_state (:407-420) at every step.
//
// Here the cache of a layer is append-only: step s writes one slab cache[s] = [R, 3D] (q | k | v of
// every hypothesis alive at step s, R = the hypothesis count at step 0) and is never copied or gathered
// afterwards.  A beam reorder moves the int32 ancestry table instead: anc[s, b] is the cache row that
// holds, at step s, the ancestor of hypothesis b, and the kernel gathers the keys through it.  The
// per-step key-padding bytes live with the cache rows ([T_cap, R]) and are addressed the same way.
//
//   CTA   = one query row (i, b), warp <-> head: the H warps share the key-row list (ancestry lookup and
//           padding folded in once, in shared memory) and nothing else, so no cross-warp reduction.
//   scores  lane <-> key: a lane pulls the key's head row (bf16: 128 bytes, 8 x LDG.128; fp32: 256 bytes,
//           16 x LDG.128) into registers as 64 floats and dots it with the query broadcast from shared memory
//   softmax fp32 over the warp's row in shared memory; a masked key's weight is exactly 0
//   p.V     the two half-warps take alternate keys, a lane 4 output dims (8 keys in flight per half-warp),
//           and the halves are added once at the end (fixed order)
//   weights per head straight from shared memory; the head average the reference returns
//           (multihead_attention.py:355-362) is a fixed-order sum over the H rows in shared memory.
//
// One kernel body serves both operand types (template on the element type T): bf16 q / cache / out
// (fbkst_dec_self_attn_fwd) and fp32 (fbkst_dec_self_attn_fwd_f32).  Only loads and stores differ.
#include <math.h>

#include <cuda_bf16.h>

#include "host_common.h"

namespace fbkst {
namespace {

constexpr int SA_HD = 64;
constexpr int SA_MAX_H = 16;
constexpr size_t SA_MAX_SMEM = 200 * 1024;

__device__ __forceinline__ float sa_bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float sa_bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

// two consecutive elements as floats (4-byte aligned for bf16, 8-byte for fp32)
__device__ __forceinline__ float2 sa_ld2(const __nv_bfloat16* p) {
  const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(p));
  return make_float2(sa_bf16_lo(w), sa_bf16_hi(w));
}
__device__ __forceinline__ float2 sa_ld2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }

// four consecutive elements as floats (8-byte aligned for bf16, 16-byte for fp32)
__device__ __forceinline__ float4 sa_ld4(const __nv_bfloat16* p) {
  const uint2 w = __ldg(reinterpret_cast<const uint2*>(p));
  return make_float4(sa_bf16_lo(w.x), sa_bf16_hi(w.x), sa_bf16_lo(w.y), sa_bf16_hi(w.y));
}
__device__ __forceinline__ float4 sa_ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

__device__ __forceinline__ void sa_st4(__nv_bfloat16* p, float4 v) {
  const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  uint2 w;
  w.x = *reinterpret_cast<const uint32_t*>(&a);
  w.y = *reinterpret_cast<const uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = w;
}
__device__ __forceinline__ void sa_st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// one 64-element head row (16-byte aligned) -> kf[64]
__device__ __forceinline__ void sa_ld_row(const __nv_bfloat16* p, float (&kf)[SA_HD]) {
  const uint4* kp = reinterpret_cast<const uint4*>(p);
  uint4 kr[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) kr[i] = __ldg(kp + i);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    kf[8 * i + 0] = sa_bf16_lo(kr[i].x); kf[8 * i + 1] = sa_bf16_hi(kr[i].x);
    kf[8 * i + 2] = sa_bf16_lo(kr[i].y); kf[8 * i + 3] = sa_bf16_hi(kr[i].y);
    kf[8 * i + 4] = sa_bf16_lo(kr[i].z); kf[8 * i + 5] = sa_bf16_hi(kr[i].z);
    kf[8 * i + 6] = sa_bf16_lo(kr[i].w); kf[8 * i + 7] = sa_bf16_hi(kr[i].w);
  }
}
__device__ __forceinline__ void sa_ld_row(const float* p, float (&kf)[SA_HD]) {
  const float4* kp = reinterpret_cast<const float4*>(p);
#pragma unroll
  for (int i = 0; i < SA_HD / 4; ++i) {
    const float4 v = __ldg(kp + i);
    kf[4 * i + 0] = v.x; kf[4 * i + 1] = v.y; kf[4 * i + 2] = v.z; kf[4 * i + 3] = v.w;
  }
}

// key-row list [n_keys] int, then per head: query [64] and scores / probabilities [n_keys] floats
__host__ __device__ inline int sa_keys_padded(int n_keys) { return (n_keys + 3) & ~3; }
inline size_t sa_smem_bytes(int n_keys, int H) {
  return sizeof(int) * sa_keys_padded(n_keys) + sizeof(float) * (size_t)H * (SA_HD + sa_keys_padded(n_keys));
}

}  // namespace

template <typename T>
__global__ void __launch_bounds__(SA_MAX_H * 32)
    dec_self_attn_kernel(const T* __restrict__ q, long long ldq, const T* __restrict__ cache,
                         const int* __restrict__ anc, const uint8_t* __restrict__ pad, T* __restrict__ out,
                         float* __restrict__ attn_w, int w_mode, int causal, int n_keys, int R, int bsz,
                         int tgt_len, int H) {
  extern __shared__ __align__(16) uint8_t sa_raw[];
  const int nk4 = sa_keys_padded(n_keys);
  int* s_row = reinterpret_cast<int*>(sa_raw);       // [nk4] cache row of key s; -1: masked, never read
  float* s_q = reinterpret_cast<float*>(s_row + nk4);  // [H][64]
  float* s_p = s_q + H * SA_HD;                        // [H][nk4]
  const int D = H * SA_HD;
  const size_t ld = (size_t)3 * D;                     // cache row pitch: q | k | v
  const int qi = blockIdx.x;                           // query row i * bsz + b
  const int i = qi / bsz, b = qi - i * bsz;
  const int h = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_vis = causal ? i + 1 : n_keys;           // keys 0 .. n_vis-1 are visible to this query

  for (int s = threadIdx.x; s < n_vis; s += blockDim.x) {
    int row = anc != nullptr ? __ldg(anc + (size_t)s * bsz + b) : b;
    // an ancestry entry outside [0, R) addresses no cache row: the key is treated as masked
    if (row < 0 || row >= R || (pad != nullptr && pad[(size_t)s * R + row])) row = -1;
    s_row[s] = row;
  }
  reinterpret_cast<float2*>(s_q + h * SA_HD)[lane] = sa_ld2(q + (size_t)qi * ldq + h * SA_HD + 2 * lane);
  __syncthreads();

  // ---- scores: lane <-> key
  float* p = s_p + (size_t)h * nk4;
  {
    const float4* qp = reinterpret_cast<const float4*>(s_q + h * SA_HD);
    const T* kcol = cache + D + h * SA_HD;
    for (int s = lane; s < n_vis; s += 32) {
      const int row = s_row[s];
      float sc = -INFINITY;  // multihead_attention.py:330-335
      if (row >= 0) {
        float kf[SA_HD];
        sa_ld_row(kcol + ((size_t)s * R + row) * ld, kf);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int c = 0; c < SA_HD / 4; ++c) {
          const float4 qv = qp[c];  // broadcast
          a0 = fmaf(qv.x, kf[4 * c + 0], a0);
          a1 = fmaf(qv.y, kf[4 * c + 1], a1);
          a2 = fmaf(qv.z, kf[4 * c + 2], a2);
          a3 = fmaf(qv.w, kf[4 * c + 3], a3);
        }
        sc = (a0 + a1) + (a2 + a3);
      }
      p[s] = sc;
    }
  }
  __syncwarp();

  // ---- softmax (fp32, like utils.softmax on the float scores: :340-343), normalised in place
  {
    float mx = -INFINITY;
    for (int s = lane; s < n_vis; s += 32) mx = fmaxf(mx, p[s]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.0f;
    if (mx > -INFINITY) {
      for (int s = lane; s < n_vis; s += 32) {
        const float e = exp2f((p[s] - mx) * 1.4426950408889634f);  // a masked key: exp2(-inf) = 0 exactly
        p[s] = e;
        sum += e;
      }
    } else {  // every visible key masked (the reference would produce NaN): zero weights and output
      for (int s = lane; s < n_vis; s += 32) p[s] = 0.0f;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = sum > 0.0f ? 1.0f / sum : 0.0f;
    for (int s = lane; s < n_vis; s += 32) p[s] *= inv;
  }
  __syncwarp();

  // ---- p.V: half-warp `half` takes keys half, half + 2, ...; lane 4 output dims
  {
    const int half = lane >> 4, c4 = (lane & 15) * 4;
    const T* vcol = cache + 2 * D + h * SA_HD + c4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int s = half;
    // a masked key has p = 0: its value is read from row 0 of its step (always written) instead of branching
    for (; s + 14 < n_vis; s += 16) {
      float4 vv[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int key = s + 2 * k;
        vv[k] = sa_ld4(vcol + ((size_t)key * R + max(s_row[key], 0)) * ld);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float pk = p[s + 2 * k];
        acc.x = fmaf(pk, vv[k].x, acc.x); acc.y = fmaf(pk, vv[k].y, acc.y);
        acc.z = fmaf(pk, vv[k].z, acc.z); acc.w = fmaf(pk, vv[k].w, acc.w);
      }
    }
    for (; s < n_vis; s += 2) {
      const float4 v = sa_ld4(vcol + ((size_t)s * R + max(s_row[s], 0)) * ld);
      const float pk = p[s];
      acc.x = fmaf(pk, v.x, acc.x); acc.y = fmaf(pk, v.y, acc.y);
      acc.z = fmaf(pk, v.z, acc.z); acc.w = fmaf(pk, v.w, acc.w);
    }
    acc.x += __shfl_xor_sync(0xffffffffu, acc.x, 16);
    acc.y += __shfl_xor_sync(0xffffffffu, acc.y, 16);
    acc.z += __shfl_xor_sync(0xffffffffu, acc.z, 16);
    acc.w += __shfl_xor_sync(0xffffffffu, acc.w, 16);
    if (half == 0) sa_st4(out + (size_t)qi * D + h * SA_HD + c4, acc);
  }

  // ---- weights over all n_keys positions (invisible future keys: 0)
  if (w_mode == 2) {  // per head [H, bsz, tgt_len, n_keys]
    float* w = attn_w + (((size_t)h * bsz + b) * tgt_len + i) * n_keys;
    for (int s = lane; s < n_keys; s += 32) w[s] = s < n_vis ? p[s] : 0.0f;
  } else if (w_mode == 1) {  // mean over heads [bsz, tgt_len, n_keys], fixed order
    __syncthreads();
    float* w = attn_w + ((size_t)b * tgt_len + i) * n_keys;
    const float invH = 1.0f / (float)H;
    for (int s = threadIdx.x; s < n_keys; s += blockDim.x) {
      float a = 0.0f;
      if (s < n_vis)
        for (int hh = 0; hh < H; ++hh) a += s_p[(size_t)hh * nk4 + s];
      w[s] = a * invH;
    }
  }
}

// The launch behind both entry points: T is the element type of q, cache and out.
template <typename T>
int dec_self_attn_launch(const char* name, const void* q, int64_t ldq, const void* cache, const int32_t* anc,
                         const uint8_t* key_padding, void* out, float* attn_w, int w_mode, int mode, int n_keys,
                         int R, int bsz, int tgt_len, int H, fbkst_stream_t stream) {
  FBKST_REQUIRE(q && cache && out, "%s: null pointer", name);
  FBKST_REQUIRE(n_keys >= 1 && R >= 1 && bsz >= 1 && tgt_len >= 1,
                "%s: empty problem (n_keys=%d R=%d bsz=%d tgt_len=%d)", name, n_keys, R, bsz, tgt_len);
  FBKST_REQUIRE(bsz <= R, "%s: %d hypothesis rows but the cache holds %d rows per step", name, bsz, R);
  FBKST_REQUIRE(H >= 1 && H <= SA_MAX_H, "%s: heads must be in [1,16] (head_dim is 64), got %d", name, H);
  FBKST_REQUIRE(mode >= FBKST_SA_INCREMENTAL && mode <= FBKST_SA_CAUSAL, "%s: unknown mode %d", name, mode);
  FBKST_REQUIRE(mode != FBKST_SA_INCREMENTAL || tgt_len == 1, "%s: incremental mode takes one query per row, got %d",
                name, tgt_len);
  FBKST_REQUIRE(mode == FBKST_SA_INCREMENTAL || n_keys == tgt_len,
                "%s: full / causal mode needs n_keys == tgt_len (%d != %d)", name, n_keys, tgt_len);
  FBKST_REQUIRE(w_mode >= 0 && w_mode <= 2 && (w_mode == 0 || attn_w), "%s: bad attention-weight mode", name);
  FBKST_REQUIRE(ldq >= (int64_t)H * SA_HD && ldq % 2 == 0, "%s: query row pitch %lld too small or odd", name,
                (long long)ldq);
  FBKST_REQUIRE((reinterpret_cast<uintptr_t>(q) & (2 * sizeof(T) - 1)) == 0 &&
                    (reinterpret_cast<uintptr_t>(cache) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                "%s: q must be aligned to two elements, cache and out to 16 bytes", name);
  const size_t smem = sa_smem_bytes(n_keys, H);
  FBKST_REQUIRE(smem <= SA_MAX_SMEM, "%s: %d keys x %d heads do not fit in shared memory", name, n_keys, H);
  const long long ctas = (long long)bsz * tgt_len;
  FBKST_REQUIRE(ctas <= 0x7fffffffLL, "%s: problem too large", name);
  static PerDeviceFlag configured;  // one per instantiation
  if (smem > 48 * 1024 && !configured) {
    FBKST_CHECK_CUDA(
        cudaFuncSetAttribute(dec_self_attn_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SA_MAX_SMEM));
    configured = true;
  }
  dec_self_attn_kernel<T><<<(unsigned)ctas, H * 32, smem, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const T*>(q), (long long)ldq, static_cast<const T*>(cache), anc, key_padding, static_cast<T*>(out),
      w_mode ? attn_w : nullptr, w_mode, mode == FBKST_SA_CAUSAL ? 1 : 0, n_keys, R, bsz, tgt_len, H);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace fbkst

extern "C" int fbkst_dec_self_attn_fwd(const void* q, int64_t ldq, const void* cache, const int32_t* anc,
                                       const uint8_t* key_padding, void* out, float* attn_w, int w_mode, int mode,
                                       int n_keys, int R, int bsz, int tgt_len, int H, fbkst_stream_t stream) {
  return fbkst::dec_self_attn_launch<__nv_bfloat16>("dec_self_attn_fwd", q, ldq, cache, anc, key_padding, out, attn_w,
                                                    w_mode, mode, n_keys, R, bsz, tgt_len, H, stream);
}

extern "C" int fbkst_dec_self_attn_fwd_f32(const float* q, int64_t ldq, const float* cache, const int32_t* anc,
                                           const uint8_t* key_padding, float* out, float* attn_w, int w_mode,
                                           int mode, int n_keys, int R, int bsz, int tgt_len, int H,
                                           fbkst_stream_t stream) {
  return fbkst::dec_self_attn_launch<float>("dec_self_attn_fwd_f32", q, ldq, cache, anc, key_padding, out, attn_w,
                                            w_mode, mode, n_keys, R, bsz, tgt_len, H, stream);
}
