// HBM-bound kernels of the path: fbank CMVN, LayerNorm, sinusoidal table, padding mask, and the
// weight-format preparation kernels; also the conv1 entry points (the kernel is in conv1_tcgen05.cu).
#include <math.h>

#include <cuda_fp16.h>

#include "host_common.h"
#include "ptx.cuh"

namespace fbkst {

// ------------------------------------------------------------------ CMVN (a1)
// Pass 1: per (utterance, feature) sum and sum of squares in fp64 (unbiased variance needs
// sumsq - sum^2/n; fp64 keeps the cancellation harmless).  grid = (chunks, B).
// `starts` (optional): x is a RAGGED buffer [sum(len), F] and utterance b begins at frame starts[b]
// (device collater, a2 of the "next" rows: data/collaters.py:43-56); otherwise x is padded [B,T,F].
__global__ void cmvn_stats_kernel(const float* __restrict__ x, const long long* __restrict__ starts,
                                  const int* __restrict__ lengths, double* __restrict__ ws, int T, int F,
                                  int rows_per_block) {
  extern __shared__ double sred[];  // [2][blockDim.x]
  const int b = blockIdx.y;
  const int len = min(lengths[b], T);
  const int t0 = blockIdx.x * rows_per_block;
  const int t1 = min(t0 + rows_per_block, len);
  const int groups = blockDim.x / F;  // row groups handled concurrently
  const int f = threadIdx.x % F, g = threadIdx.x / F;
  double s = 0.0, ss = 0.0;
  if (g < groups) {
    const float* xp = x + (starts ? (size_t)starts[b] : (size_t)b * T) * F + f;
    for (int t = t0 + g; t < t1; t += groups) {
      const double v = (double)__ldg(xp + (size_t)t * F);
      s += v;
      ss += v * v;
    }
  }
  sred[threadIdx.x] = s;
  sred[blockDim.x + threadIdx.x] = ss;
  __syncthreads();
  if (threadIdx.x < F) {
    double a = 0.0, c = 0.0;
    for (int k = 0; k < groups; ++k) {
      a += sred[k * F + threadIdx.x];
      c += sred[blockDim.x + k * F + threadIdx.x];
    }
    if (t0 < t1) {
      atomicAdd(&ws[((size_t)b * F + threadIdx.x) * 2 + 0], a);
      atomicAdd(&ws[((size_t)b * F + threadIdx.x) * 2 + 1], c);
    }
  }
}

// Pass 2: y = (x - mean) * inv with the reference's eps rule (data_utils.py:15-19): if ANY
// feature of the utterance has var < 1e-8, inv = 1/(sqrt(var)+1e-8) for all features.
// With `starts` the input is ragged and the output padded (collate + normalise in one pass); with
// ws == nullptr nothing is normalised (pure zero-padded collate).
__global__ void cmvn_apply_kernel(const float* __restrict__ x, const long long* __restrict__ starts,
                                  float* __restrict__ y, const int* __restrict__ lengths,
                                  const double* __restrict__ ws, int T, int F, int rows_per_block) {
  extern __shared__ float sstat[];  // mean[F], inv[F]
  const int b = blockIdx.y;
  const int len = min(lengths[b], T);
  int small = 0;
  float mean = 0.f, var = 0.f;
  if (threadIdx.x < F && ws != nullptr) {
    const double n = (double)len;
    const double s = ws[((size_t)b * F + threadIdx.x) * 2 + 0];
    const double ss = ws[((size_t)b * F + threadIdx.x) * 2 + 1];
    const double m = s / n;
    double v = (ss - s * m) / (n - 1.0);
    if (v < 0.0) v = 0.0;
    mean = (float)m;
    var = (float)v;
    small = var < 1e-8f;
  }
  const int any_small = __syncthreads_or(small);
  if (threadIdx.x < F) {
    sstat[threadIdx.x] = mean;
    sstat[F + threadIdx.x] =
        ws == nullptr ? 1.0f : (any_small ? 1.0f / (sqrtf(var) + 1e-8f) : 1.0f / sqrtf(var));
  }
  __syncthreads();
  const int t0 = blockIdx.x * rows_per_block;
  const int t1 = min(t0 + rows_per_block, T);
  const size_t base = ((size_t)b * T + t0) * F;
  const size_t ibase = starts ? ((size_t)starts[b] + t0) * F : base;
  const int n = (t1 - t0) * F;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int t = t0 + i / F, f = i % F;
    y[base + i] = (t < len) ? (__ldg(x + ibase + i) - sstat[f]) * sstat[F + f] : 0.0f;
  }
}

// float4 versions of the two CMVN passes for F % 4 == 0 (every reference recipe: F = 40 / 80): thread <->
// (feature quad, row group), no integer division in the row loops, 16-byte loads and stores.  Same fp64
// statistics, same eps rule; the scalar kernels above serve any other F.
__global__ void __launch_bounds__(256)
    cmvn_stats4_kernel(const float* __restrict__ x, const long long* __restrict__ starts,
                       const int* __restrict__ lengths, double* __restrict__ ws, int T, int F,
                       int rows_per_block) {
  extern __shared__ double sred[];  // [2][RG][F]
  const int Q = F >> 2, RG = blockDim.x / Q;
  const int b = blockIdx.y;
  const int len = min(lengths[b], T);
  const int t0 = blockIdx.x * rows_per_block;
  const int t1 = min(t0 + rows_per_block, len);
  const int q = threadIdx.x % Q, rg = threadIdx.x / Q;
  double s[4] = {0.0, 0.0, 0.0, 0.0}, ss[4] = {0.0, 0.0, 0.0, 0.0};
  if (rg < RG) {
    const float4* xp = reinterpret_cast<const float4*>(x + (starts ? (size_t)starts[b] : (size_t)b * T) * F) + q;
#pragma unroll 4
    for (int t = t0 + rg; t < t1; t += RG) {
      const float4 v = __ldg(xp + (size_t)t * Q);
      s[0] += (double)v.x; ss[0] += (double)v.x * (double)v.x;
      s[1] += (double)v.y; ss[1] += (double)v.y * (double)v.y;
      s[2] += (double)v.z; ss[2] += (double)v.z * (double)v.z;
      s[3] += (double)v.w; ss[3] += (double)v.w * (double)v.w;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      sred[rg * F + q * 4 + j] = s[j];
      sred[(RG + rg) * F + q * 4 + j] = ss[j];
    }
  }
  __syncthreads();
  if (threadIdx.x < F && t0 < t1) {
    double a = 0.0, c = 0.0;
    for (int k = 0; k < RG; ++k) {
      a += sred[k * F + threadIdx.x];
      c += sred[(RG + k) * F + threadIdx.x];
    }
    atomicAdd(&ws[((size_t)b * F + threadIdx.x) * 2 + 0], a);
    atomicAdd(&ws[((size_t)b * F + threadIdx.x) * 2 + 1], c);
  }
}

__global__ void __launch_bounds__(256)
    cmvn_apply4_kernel(const float* __restrict__ x, const long long* __restrict__ starts,
                       float* __restrict__ y, const int* __restrict__ lengths,
                       const double* __restrict__ ws, int T, int F, int rows_per_block) {
  extern __shared__ float sstat[];  // mean[F], inv[F]
  const int b = blockIdx.y;
  const int len = min(lengths[b], T);
  int small = 0;
  float mean = 0.f, var = 0.f;
  if (threadIdx.x < F && ws != nullptr) {
    const double n = (double)len;
    const double s = ws[((size_t)b * F + threadIdx.x) * 2 + 0];
    const double ss = ws[((size_t)b * F + threadIdx.x) * 2 + 1];
    const double m = s / n;
    double v = (ss - s * m) / (n - 1.0);
    if (v < 0.0) v = 0.0;
    mean = (float)m;
    var = (float)v;
    small = var < 1e-8f;
  }
  const int any_small = __syncthreads_or(small);
  if (threadIdx.x < F) {
    sstat[threadIdx.x] = mean;
    sstat[F + threadIdx.x] =
        ws == nullptr ? 1.0f : (any_small ? 1.0f / (sqrtf(var) + 1e-8f) : 1.0f / sqrtf(var));
  }
  __syncthreads();
  const int Q = F >> 2, RG = blockDim.x / Q;
  const int q = threadIdx.x % Q, rg = threadIdx.x / Q;
  if (rg >= RG) return;
  const float4 m4 = reinterpret_cast<const float4*>(sstat)[q];
  const float4 i4 = reinterpret_cast<const float4*>(sstat + F)[q];
  const int t0 = blockIdx.x * rows_per_block;
  const int t1 = min(t0 + rows_per_block, T);
  const float4* xp = reinterpret_cast<const float4*>(x + (starts ? (size_t)starts[b] : (size_t)b * T) * F) + q;
  float4* yp = reinterpret_cast<float4*>(y + (size_t)b * T * F) + q;
#pragma unroll 4
  for (int t = t0 + rg; t < t1; t += RG) {
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t < len) {
      const float4 v = __ldg(xp + (size_t)t * Q);
      o.x = (v.x - m4.x) * i4.x;
      o.y = (v.y - m4.y) * i4.y;
      o.z = (v.z - m4.z) * i4.z;
      o.w = (v.w - m4.w) * i4.w;
    }
    yp[(size_t)t * Q] = o;
  }
}

// ------------------------------------------------------------- LayerNorm (a8)
// One warp per row, the row held in registers (NV float4 per lane), two-pass variance.
template <int NV>
__global__ void __launch_bounds__(256)
    layernorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                     const float* __restrict__ beta, void* __restrict__ y, int out_f32, int M,
                     float eps, const int* __restrict__ m_limit, int m_limit_mult) {
  constexpr int D = NV * 128;
  pdl_launch_dependents();
  pdl_wait();
  if (m_limit != nullptr) M = min(M, __ldg(m_limit) * m_limit_mult);
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const int lane = threadIdx.x & 31;
  const float4* xp = reinterpret_cast<const float4*>(x + (size_t)row * D);
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i] = xp[i * 32 + lane];
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  const float mean = warp_sum(s) * (1.0f / D);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / D) + eps);
  const float4* gp = reinterpret_cast<const float4*>(gamma);
  const float4* bp = reinterpret_cast<const float4*>(beta);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float4 g = __ldg(gp + i * 32 + lane), b = __ldg(bp + i * 32 + lane);
    float4 o;
    o.x = (v[i].x - mean) * rstd * g.x + b.x;
    o.y = (v[i].y - mean) * rstd * g.y + b.y;
    o.z = (v[i].z - mean) * rstd * g.z + b.z;
    o.w = (v[i].w - mean) * rstd * g.w + b.w;
    if (out_f32) {
      reinterpret_cast<float4*>(reinterpret_cast<float*>(y) + (size_t)row * D)[i * 32 + lane] = o;
    } else {
      reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(y) + (size_t)row * D)[i * 32 + lane] =
          make_uint2(pack_bf16x2(o.x, o.y), pack_bf16x2(o.z, o.w));
    }
  }
}

// Row statistics + bf16 copy for the folded LayerNorm (gemm2_tcgen05.cu): for an x that does not
// come out of a residual GEMM (fc3 output, CTC-compressed rows) this produces what that epilogue
// would have: xb = bf16(x) and, per row and 128-column slice, (mean, M2) of the slice.
template <int NV>
__global__ void __launch_bounds__(256)
    row_stats_cast_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ xb,
                          float2* __restrict__ stats, int M, const int* __restrict__ m_limit,
                          int m_limit_mult) {
  constexpr int D = NV * 128;
  pdl_launch_dependents();
  pdl_wait();
  if (m_limit != nullptr) M = min(M, __ldg(m_limit) * m_limit_mult);
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= M) return;
  const int lane = threadIdx.x & 31;
  const float4* xp = reinterpret_cast<const float4*>(x + (size_t)row * D);
  float4 v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = xp[i * 32 + lane];
  float keep_mean = 0.f, keep_m2 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float mean = warp_sum((v[i].x + v[i].y) + (v[i].z + v[i].w)) * (1.0f / 128.0f);
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    const float m2 = warp_sum((a * a + b * b) + (c * c + d * d));
    if (lane == i) {
      keep_mean = mean;
      keep_m2 = m2;
    }
    reinterpret_cast<uint2*>(xb + (size_t)row * D)[i * 32 + lane] =
        make_uint2(pack_bf16x2(v[i].x, v[i].y), pack_bf16x2(v[i].z, v[i].w));
  }
  if (lane < NV) stats[(size_t)row * NV + lane] = make_float2(keep_mean, keep_m2);
}

// fc3 epilogue that is not a GEMM epilogue (conv_transformer.py:225-229): the fc3 GEMM writes relu(a W^T
// + b) in the conv layout's row order (b, t); this kernel moves row (b, t) to the time-major row t*B + b,
// adds the sinusoidal position (row t+1 of the table inside the utterance, the padding row 0 beyond
// its length) and emits what row_stats_cast would: fp32 x, bf16 x and the per-slice LayerNorm statistics
// of the first layer.  One warp per row: 2 KB coalesced reads and writes.  Measured (ncu, cfg2): CTA-pair
// GEMM 21.7 us + this kernel 18.6 us, against 52.3 us for the single-CTA GEMM with the row-remapping
// thread-per-row epilogue + 11.3 us for the separate row_stats_cast pass.
template <int NV>
__global__ void __launch_bounds__(256)
    embed_remap_stats_kernel(const float* __restrict__ src, const float* __restrict__ table,
                             long long ld_table, const int* __restrict__ lengths,
                             float* __restrict__ x, __nv_bfloat16* __restrict__ xb,
                             float2* __restrict__ stats, int L, int B) {
  constexpr int D = NV * 128;
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);  // t * B + b
  if (row >= L * B) return;
  const int lane = threadIdx.x & 31;
  const int t = row / B, b = row - t * B;
  const float4* sp = reinterpret_cast<const float4*>(src + ((size_t)b * L + t) * D);
  float4 v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = __ldg(sp + i * 32 + lane);
  if (table != nullptr) {
    const int prow = (t < __ldg(lengths + b)) ? t + 1 : 0;
    const float4* tp = reinterpret_cast<const float4*>(table + (size_t)prow * ld_table);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float4 p = __ldg(tp + i * 32 + lane);
      v[i].x += p.x; v[i].y += p.y; v[i].z += p.z; v[i].w += p.w;
    }
  }
  float keep_mean = 0.f, keep_m2 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float mean = warp_sum((v[i].x + v[i].y) + (v[i].z + v[i].w)) * (1.0f / 128.0f);
    const float a = v[i].x - mean, bb = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    const float m2 = warp_sum((a * a + bb * bb) + (c * c + d * d));
    if (lane == i) {
      keep_mean = mean;
      keep_m2 = m2;
    }
    reinterpret_cast<float4*>(x + (size_t)row * D)[i * 32 + lane] = v[i];
    reinterpret_cast<uint2*>(xb + (size_t)row * D)[i * 32 + lane] =
        make_uint2(pack_bf16x2(v[i].x, v[i].y), pack_bf16x2(v[i].z, v[i].w));
  }
  if (lane < NV) stats[(size_t)row * NV + lane] = make_float2(keep_mean, keep_m2);
}

// ------------------------------------------------------ sinusoidal table (a4)
__global__ void sinusoidal_table_kernel(float* __restrict__ table, int rows, int D) {
  const int half = D / 2;
  const float step = -(logf(10000.0f) / (float)(half - 1));
  const long long total = (long long)rows * D;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int p = (int)(i / D), c = (int)(i % D);
    float val = 0.0f;
    if (p > 0 && c < 2 * half) {
      const int k = c < half ? c : c - half;
      const float ang = (float)p * expf((float)k * step);
      val = c < half ? sinf(ang) : cosf(ang);
    }
    table[i] = val;
  }
}

// ----------------------------------------------------------- padding mask (a5)
__global__ void lengths_to_mask_kernel(const int* __restrict__ lengths, uint8_t* __restrict__ mask,
                                       int* __restrict__ any_pad, int B, int L) {
  const int total = B * L;
  int pad_seen = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / L, t = i - b * L;
    const uint8_t m = t >= lengths[b];
    mask[i] = m;
    pad_seen |= m;
  }
  if (__syncthreads_or(pad_seen) && threadIdx.x == 0) atomicOr(any_pad, 1);
}

// lengths after `times` stride-2 convolutions: n -> ceil(n / 2) each (conv_transformer.py:213), from the
// int64 (fairseq) or int32 lengths wherever they live on the device: no host round trip for shape logic
__global__ void subsample_lengths_kernel(const void* __restrict__ in, int in_is_i64, int* __restrict__ out,
                                         int B, int times) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  long long n = in_is_i64 ? reinterpret_cast<const long long*>(in)[b]
                          : (long long)reinterpret_cast<const int*>(in)[b];
  for (int i = 0; i < times; ++i) n = (n + 1) >> 1;
  out[b] = (int)n;
}

// ----------------------------------------------------------- weight preparation
__global__ void cast_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                 long long n, float scale) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x)
    dst[i] = __float2bfloat16_rn(src[i] * scale);
}
__device__ __forceinline__ __half f2h_sat(float x) {
  return __float2half_rn(fminf(fmaxf(x, -65504.0f), 65504.0f));
}
__global__ void prep_conv2_weight_kernel(const float* __restrict__ w, __half* __restrict__ o,
                                         int C) {
  const int total = 9 * C * C;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int ci = i % C, co = (i / C) % C, tap = i / (C * C);
    o[i] = f2h_sat(w[((size_t)co * C + ci) * 9 + tap]);
  }
}
__global__ void prep_fc3_weight_kernel(const float* __restrict__ w, __half* __restrict__ o,
                                       int D, int C, int F2) {
  const long long total = (long long)D * C * F2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C), f = (int)((i / C) % F2), d = (int)(i / ((long long)C * F2));
    o[i] = f2h_sat(w[((size_t)d * C + c) * F2 + f]);
  }
}
__global__ void prep_bn_affine_kernel(const float* gamma, const float* beta, const float* mean,
                                      const float* var, float eps, float* scale, float* shift,
                                      int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    const float s = gamma[c] / sqrtf(var[c] + eps);
    scale[c] = s;
    shift[c] = beta[c] - mean[c] * s;
  }
}

static inline int grid_for(long long n, int block, int cap_mult = 8) {
  long long g = (n + block - 1) / block;
  const long long cap = (long long)num_sms() * cap_mult;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace fbkst

using namespace fbkst;

extern "C" int fbkst_cmvn_f32(const float* x, float* y, const int32_t* lengths, int B, int T, int F,
                              double* workspace, fbkst_stream_t stream) {
  FBKST_REQUIRE(x && y && lengths && workspace, "fbkst_cmvn_f32: null pointer");
  FBKST_REQUIRE(B > 0 && T > 0 && F > 0 && F <= 256, "fbkst_cmvn_f32: bad shape B=%d T=%d F=%d", B,
                T, F);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  FBKST_CHECK_CUDA(cudaMemsetAsync(workspace, 0, sizeof(double) * 2 * B * F, st));
  const int rows = 128;
  dim3 grid((T + rows - 1) / rows, B);
  if (F % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0) {
    const int RG = 256 / (F / 4);
    cmvn_stats4_kernel<<<grid, 256, 2 * RG * F * sizeof(double), st>>>(x, nullptr, lengths, workspace, T, F, rows);
    cmvn_apply4_kernel<<<grid, 256, 2 * F * sizeof(float), st>>>(x, nullptr, y, lengths, workspace, T, F, rows);
  } else {
    cmvn_stats_kernel<<<grid, 256, 2 * 256 * sizeof(double), st>>>(x, nullptr, lengths, workspace, T, F, rows);
    cmvn_apply_kernel<<<grid, 256, 2 * F * sizeof(float), st>>>(x, nullptr, y, lengths, workspace, T, F, rows);
  }
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_collate_cmvn_f32(const float* packed, const int64_t* starts, const int32_t* lengths,
                                      float* out, int B, int T, int F, int normalize, double* workspace,
                                      fbkst_stream_t stream) {
  FBKST_REQUIRE(packed && starts && lengths && out, "fbkst_collate_cmvn_f32: null pointer");
  FBKST_REQUIRE(!normalize || workspace, "fbkst_collate_cmvn_f32: normalisation needs a workspace");
  FBKST_REQUIRE(B > 0 && T > 0 && F > 0 && F <= 256, "fbkst_collate_cmvn_f32: bad shape B=%d T=%d F=%d",
                B, T, F);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int rows = 128;
  dim3 grid((T + rows - 1) / rows, B);
  const long long* sp = reinterpret_cast<const long long*>(starts);
  const bool vec4 = F % 4 == 0 && (reinterpret_cast<uintptr_t>(packed) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(out) & 15) == 0;
  if (normalize) {
    FBKST_CHECK_CUDA(cudaMemsetAsync(workspace, 0, sizeof(double) * 2 * B * F, st));
    if (vec4)
      cmvn_stats4_kernel<<<grid, 256, 2 * (256 / (F / 4)) * F * sizeof(double), st>>>(packed, sp, lengths,
                                                                                    workspace, T, F, rows);
    else
      cmvn_stats_kernel<<<grid, 256, 2 * 256 * sizeof(double), st>>>(packed, sp, lengths, workspace, T, F, rows);
  }
  if (vec4)
    cmvn_apply4_kernel<<<grid, 256, 2 * F * sizeof(float), st>>>(packed, sp, out, lengths,
                                                                normalize ? workspace : nullptr, T, F, rows);
  else
    cmvn_apply_kernel<<<grid, 256, 2 * F * sizeof(float), st>>>(packed, sp, out, lengths,
                                                               normalize ? workspace : nullptr, T, F, rows);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_conv1_relu_bn(const float* x, const float* w, const float* bias,
                                   const float* bn_scale, const float* bn_shift, void* y, int B,
                                   int T, int F, int C, fbkst_stream_t stream) {
  FBKST_REQUIRE(x && w && bias && bn_scale && bn_shift && y, "fbkst_conv1_relu_bn: null pointer");
  FBKST_REQUIRE(C == 64 || C == 128, "fbkst_conv1_relu_bn: C must be 64 or 128 (got %d)", C);
  FBKST_REQUIRE(B > 0 && T > 0 && F > 0, "fbkst_conv1_relu_bn: bad shape");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int T1 = (T + 1) / 2, F1 = (F + 1) / 2;
  FBKST_REQUIRE((long long)B * T1 * F1 < (1ll << 31), "fbkst_conv1_relu_bn: too many pixels");
  return conv1_tc_dispatch(x, w, bias, bn_scale, bn_shift, y, B, T, F, C, T1, F1, st);
}

extern "C" int fbkst_layernorm(const float* x, const float* gamma, const float* beta, void* y,
                               int out_dtype, int M, int D, float eps, const int32_t* m_limit,
                               int m_limit_mult, fbkst_stream_t stream) {
  FBKST_REQUIRE(x && gamma && beta && y, "fbkst_layernorm: null pointer");
  FBKST_REQUIRE(M > 0, "fbkst_layernorm: M must be positive");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int f32 = out_dtype == FBKST_F32;
  const int grid = (M + 7) / 8;
  switch (D) {
    case 128: FBKST_CHECK_CUDA(launch_pdl(layernorm_kernel<1>, dim3(grid), dim3(256), 0, st, x, gamma, beta, y, f32, M, eps, m_limit, m_limit_mult)); break;
    case 256: FBKST_CHECK_CUDA(launch_pdl(layernorm_kernel<2>, dim3(grid), dim3(256), 0, st, x, gamma, beta, y, f32, M, eps, m_limit, m_limit_mult)); break;
    case 384: FBKST_CHECK_CUDA(launch_pdl(layernorm_kernel<3>, dim3(grid), dim3(256), 0, st, x, gamma, beta, y, f32, M, eps, m_limit, m_limit_mult)); break;
    case 512: FBKST_CHECK_CUDA(launch_pdl(layernorm_kernel<4>, dim3(grid), dim3(256), 0, st, x, gamma, beta, y, f32, M, eps, m_limit, m_limit_mult)); break;
    case 768: FBKST_CHECK_CUDA(launch_pdl(layernorm_kernel<6>, dim3(grid), dim3(256), 0, st, x, gamma, beta, y, f32, M, eps, m_limit, m_limit_mult)); break;
    case 1024: FBKST_CHECK_CUDA(launch_pdl(layernorm_kernel<8>, dim3(grid), dim3(256), 0, st, x, gamma, beta, y, f32, M, eps, m_limit, m_limit_mult)); break;
    default:
      return set_error(FBKST_ERR_ARG, "fbkst_layernorm: unsupported D=%d (128..1024, multiple of 128)", D);
  }
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_row_stats_cast(const float* x, void* xb, float* row_stats, int M, int D,
                                    const int32_t* m_limit, int m_limit_mult, fbkst_stream_t stream) {
  FBKST_REQUIRE(x && xb && row_stats, "fbkst_row_stats_cast: null pointer");
  FBKST_REQUIRE(M > 0, "fbkst_row_stats_cast: M must be positive");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int grid = (M + 7) / 8;
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(xb);
  float2* s2 = reinterpret_cast<float2*>(row_stats);
  switch (D) {
    case 128: FBKST_CHECK_CUDA(launch_pdl(row_stats_cast_kernel<1>, dim3(grid), dim3(256), 0, st, x, o, s2, M, m_limit, m_limit_mult)); break;
    case 256: FBKST_CHECK_CUDA(launch_pdl(row_stats_cast_kernel<2>, dim3(grid), dim3(256), 0, st, x, o, s2, M, m_limit, m_limit_mult)); break;
    case 384: FBKST_CHECK_CUDA(launch_pdl(row_stats_cast_kernel<3>, dim3(grid), dim3(256), 0, st, x, o, s2, M, m_limit, m_limit_mult)); break;
    case 512: FBKST_CHECK_CUDA(launch_pdl(row_stats_cast_kernel<4>, dim3(grid), dim3(256), 0, st, x, o, s2, M, m_limit, m_limit_mult)); break;
    case 768: FBKST_CHECK_CUDA(launch_pdl(row_stats_cast_kernel<6>, dim3(grid), dim3(256), 0, st, x, o, s2, M, m_limit, m_limit_mult)); break;
    case 1024: FBKST_CHECK_CUDA(launch_pdl(row_stats_cast_kernel<8>, dim3(grid), dim3(256), 0, st, x, o, s2, M, m_limit, m_limit_mult)); break;
    default:
      return set_error(FBKST_ERR_ARG, "fbkst_row_stats_cast: unsupported D=%d (128..1024, multiple of 128)", D);
  }
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_embed_remap_stats(const float* src, const float* table, int64_t ld_table,
                                       const int32_t* lengths, float* x, void* xb, float* row_stats,
                                       int L, int B, int D, fbkst_stream_t stream) {
  FBKST_REQUIRE(src && x && xb && row_stats, "fbkst_embed_remap_stats: null pointer");
  FBKST_REQUIRE(L > 0 && B > 0, "fbkst_embed_remap_stats: bad shape L=%d B=%d", L, B);
  FBKST_REQUIRE(table == nullptr || (lengths != nullptr && ld_table % 4 == 0),
                "fbkst_embed_remap_stats: a position table needs lengths and a row stride multiple of 4");
  FBKST_REQUIRE((long long)L * B < (1ll << 31), "fbkst_embed_remap_stats: too many rows");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int grid = (L * B + 7) / 8;
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(xb);
  float2* s2 = reinterpret_cast<float2*>(row_stats);
  const long long ldt = ld_table;
#define FBKST_ERS(NV) FBKST_CHECK_CUDA(launch_pdl(embed_remap_stats_kernel<NV>, dim3(grid), dim3(256), 0, st, src, table, ldt, lengths, x, o, s2, L, B))
  switch (D) {
    case 128: FBKST_ERS(1); break;
    case 256: FBKST_ERS(2); break;
    case 384: FBKST_ERS(3); break;
    case 512: FBKST_ERS(4); break;
    case 768: FBKST_ERS(6); break;
    case 1024: FBKST_ERS(8); break;
    default:
      return set_error(FBKST_ERR_ARG, "fbkst_embed_remap_stats: unsupported D=%d (128..1024, multiple of 128)", D);
  }
#undef FBKST_ERS
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_sinusoidal_table(float* table, int rows, int D, fbkst_stream_t stream) {
  FBKST_REQUIRE(table && rows > 0 && D >= 4, "fbkst_sinusoidal_table: bad arguments");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  sinusoidal_table_kernel<<<grid_for((long long)rows * D, 256), 256, 0, st>>>(table, rows, D);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_lengths_to_mask(const int32_t* lengths, uint8_t* mask, int32_t* any_pad, int B,
                                     int L, fbkst_stream_t stream) {
  FBKST_REQUIRE(lengths && mask && any_pad && B > 0 && L > 0, "fbkst_lengths_to_mask: bad arguments");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  FBKST_CHECK_CUDA(cudaMemsetAsync(any_pad, 0, sizeof(int32_t), st));
  lengths_to_mask_kernel<<<grid_for((long long)B * L, 256), 256, 0, st>>>(lengths, mask, any_pad, B, L);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_subsample_lengths(const void* lengths, int lengths_are_i64, int32_t* out, int B,
                                       int times, fbkst_stream_t stream) {
  FBKST_REQUIRE(lengths && out && B > 0 && times >= 0, "fbkst_subsample_lengths: bad arguments");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  subsample_lengths_kernel<<<(B + 127) / 128, 128, 0, st>>>(lengths, lengths_are_i64, out, B, times);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_cast_bf16(const float* src, void* dst, int64_t n, float scale,
                               fbkst_stream_t stream) {
  FBKST_REQUIRE(src && dst && n > 0, "fbkst_cast_bf16: bad arguments");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  cast_bf16_kernel<<<grid_for(n, 256), 256, 0, st>>>(src, (__nv_bfloat16*)dst, n, scale);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_prep_conv2_weight(const float* w, void* w_taps, int C, fbkst_stream_t stream) {
  FBKST_REQUIRE(w && w_taps && C > 0, "fbkst_prep_conv2_weight: bad arguments");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  prep_conv2_weight_kernel<<<grid_for(9LL * C * C, 256), 256, 0, st>>>(w, (__half*)w_taps, C);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_prep_fc3_weight(const float* w, void* w_perm, int D, int C, int F2,
                                     fbkst_stream_t stream) {
  FBKST_REQUIRE(w && w_perm && D > 0 && C > 0 && F2 > 0, "fbkst_prep_fc3_weight: bad arguments");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  prep_fc3_weight_kernel<<<grid_for((long long)D * C * F2, 256), 256, 0, st>>>(
      w, (__half*)w_perm, D, C, F2);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_prep_bn_affine(const float* gamma, const float* beta, const float* mean,
                                    const float* var, float eps, float* scale, float* shift, int C,
                                    fbkst_stream_t stream) {
  FBKST_REQUIRE(gamma && beta && mean && var && scale && shift && C > 0,
                "fbkst_prep_bn_affine: bad arguments");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  prep_bn_affine_kernel<<<(C + 127) / 128, 128, 0, st>>>(gamma, beta, mean, var, eps, scale, shift, C);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}
