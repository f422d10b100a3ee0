// Training side of the convolutional subsampling stack (scope row T; reference
// conv_transformer.py:203-214: Conv2d -> ReLU -> BatchNorm2d -> dropout(max(p, .1)), twice) -- everything
// around the tensor-core contractions.  Activations are channels-last [P, C] (P = B*T'*F' pixels, C = 64 or
// 128 channels), fp16 in the forward (see ptx.cuh idesc_f16_f32), gradients bf16.
//
//   bn_stats + bn_finalize   per-channel batch statistics over ALL pixels of the padded batch (the reference
//                            does not mask padded frames, SURVEY F5), running-stat update (momentum, unbiased
//                            variance), and the affine (scale, shift) the apply kernel uses
//   bn_apply                 y = dropout(scale[c] * relu_out + shift[c])                     fp16 -> fp16
//   bn_bwd_reduce            per-channel sums of g and g * xhat (g = dropout-backward of the incoming gradient)
//   bn_bwd_apply             dz = relu_mask * BatchNorm-backward(g)  (batch statistics or running statistics)
//   im2col_t                 conv2 wgrad operand: colT[(tap, ci), pixel] (bf16) from conv1's fp16 output
//   col2im                   conv2 dgrad: gather-sum of the <= 4 taps that reach an input pixel
//   conv1_wgrad              dW1[co, tap], db1[co]: K = 9 outer products, SIMT (HBM-bound on the gradient read)
//   conv1_dgrad              dx[b, t, f]: the gradient of the input features (attribution, input-gradient losses)
// The contractions themselves (conv2 wgrad / dgrad as GEMMs over these operands, fc3) run on the CTA-pair
// tcgen05 kernel (gemm2_tcgen05.cu).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "host_common.h"
#include "ptx.cuh"

namespace fbkst {

// ---- stateless dropout (same generator as train_elementwise.cu: Philox4x32-7, one call per column quad)
struct ConvDropout {
  float p, scale;
  uint32_t threshold, seed_lo, seed_hi, site;
};
__device__ __forceinline__ uint4 cv_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                           uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 7; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float4 cv_keep4(const ConvDropout& d, unsigned long long quad) {
  const uint4 r = cv_philox((uint32_t)quad, (uint32_t)(quad >> 32), d.site, 0x5eedu, d.seed_lo, d.seed_hi);
  return make_float4(r.x >= d.threshold ? d.scale : 0.f, r.y >= d.threshold ? d.scale : 0.f,
                     r.z >= d.threshold ? d.scale : 0.f, r.w >= d.threshold ? d.scale : 0.f);
}
static ConvDropout cv_make_dropout(float p, uint64_t seed, int site) {
  ConvDropout d;
  d.p = p;
  d.scale = p > 0.f ? 1.0f / (1.0f - p) : 1.0f;
  const double t = (double)p * 4294967296.0;
  d.threshold = t >= 4294967295.0 ? 0xffffffffu : (uint32_t)t;
  d.seed_lo = (uint32_t)seed;
  d.seed_hi = (uint32_t)(seed >> 32);
  d.site = (uint32_t)site;
  return d;
}
__device__ __forceinline__ float2 h2_to_f2(uint32_t u) {
  return __half22float2(*reinterpret_cast<const __half2*>(&u));
}
__device__ __forceinline__ float bf_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }

// ------------------------------------------------------------------ batch statistics
// thread <-> (channel quad, pixel lane); block partial (sum | sumsq) [2, C] in fp32 -> partial[block]
template <int C>
__global__ void __launch_bounds__(256)
    bn_stats_kernel(const __half* __restrict__ y, long long P, float* __restrict__ partial) {
  constexpr int Q = C / 4;        // channel quads per pixel
  constexpr int LANES = 256 / Q;  // pixels in flight per block
  __shared__ float red[LANES][2 * C + 4];
  const int q = threadIdx.x % Q, ln = threadIdx.x / Q;
  float s[4] = {0.f, 0.f, 0.f, 0.f}, ss[4] = {0.f, 0.f, 0.f, 0.f};
  for (long long px = (long long)blockIdx.x * LANES + ln; px < P; px += (long long)gridDim.x * LANES) {
    const uint2 u = *reinterpret_cast<const uint2*>(y + px * C + q * 4);
    const float2 a = h2_to_f2(u.x), b = h2_to_f2(u.y);
    s[0] += a.x; s[1] += a.y; s[2] += b.x; s[3] += b.y;
    ss[0] = fmaf(a.x, a.x, ss[0]); ss[1] = fmaf(a.y, a.y, ss[1]);
    ss[2] = fmaf(b.x, b.x, ss[2]); ss[3] = fmaf(b.y, b.y, ss[3]);
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    red[ln][q * 4 + j] = s[j];
    red[ln][C + q * 4 + j] = ss[j];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * C; i += 256) {
    float t = 0.f;
    for (int l = 0; l < LANES; ++l) t += red[l][i];
    partial[(size_t)blockIdx.x * 2 * C + i] = t;
  }
}

// partial [G, 2, C] -> mean, rstd, (scale, shift) and the running-stat update (nn.BatchNorm2d semantics:
// running = (1 - momentum) * running + momentum * batch, with the UNBIASED batch variance)
__global__ void bn_finalize_kernel(const float* __restrict__ partial, int G, int C, double count,
                                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                   float momentum, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, float* __restrict__ mean_out,
                                   float* __restrict__ rstd_out, float* __restrict__ scale,
                                   float* __restrict__ shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double s = 0.0, ss = 0.0;
  for (int g = 0; g < G; ++g) {
    s += (double)partial[(size_t)g * 2 * C + c];
    ss += (double)partial[(size_t)g * 2 * C + C + c];
  }
  const double mean = s / count;
  double var = ss / count - mean * mean;
  if (var < 0.0) var = 0.0;
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
  mean_out[c] = (float)mean;
  rstd_out[c] = rstd;
  const float sc = gamma[c] * rstd;
  scale[c] = sc;
  shift[c] = beta[c] - (float)mean * sc;
  if (running_mean != nullptr) {
    const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
    running_mean[c] = (1.0f - momentum) * running_mean[c] + momentum * (float)mean;
    running_var[c] = (1.0f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
}

// y = dropout(scale[c] * x + shift[c]); 8 channels (16 B) per thread
__global__ void __launch_bounds__(256)
    bn_apply_kernel(const __half* __restrict__ x, __half* __restrict__ y, const float* __restrict__ scale,
                    const float* __restrict__ shift, long long P, int C, ConvDropout dp) {
  const int oct = C / 8;
  const long long total = P * oct;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c0 = (int)(i % oct) * 8;
    const uint4 u = *reinterpret_cast<const uint4*>(x + i * 8);
    float v[8];
    float2 t;
    t = h2_to_f2(u.x); v[0] = t.x; v[1] = t.y;
    t = h2_to_f2(u.y); v[2] = t.x; v[3] = t.y;
    t = h2_to_f2(u.z); v[4] = t.x; v[5] = t.y;
    t = h2_to_f2(u.w); v[6] = t.x; v[7] = t.y;
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], __ldg(scale + c0 + j), __ldg(shift + c0 + j));
    if (dp.p > 0.f) {
      const float4 k0 = cv_keep4(dp, (unsigned long long)i * 2), k1 = cv_keep4(dp, (unsigned long long)i * 2 + 1);
      v[0] *= k0.x; v[1] *= k0.y; v[2] *= k0.z; v[3] *= k0.w;
      v[4] *= k1.x; v[5] *= k1.y; v[6] *= k1.z; v[7] *= k1.w;
    }
    *reinterpret_cast<uint4*>(y + i * 8) =
        make_uint4(pack_f16x2(v[0], v[1]), pack_f16x2(v[2], v[3]), pack_f16x2(v[4], v[5]), pack_f16x2(v[6], v[7]));
  }
}

// per-channel sums of g (-> dbeta) and g * xhat (-> dgamma), g = dy o keep;  partial [G, 2, C]
template <int C>
__global__ void __launch_bounds__(256)
    bn_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ dy, const __half* __restrict__ xr,
                         const float* __restrict__ mean, const float* __restrict__ rstd, long long P,
                         float* __restrict__ partial, ConvDropout dp) {
  constexpr int Q = C / 4;
  constexpr int LANES = 256 / Q;
  __shared__ float red[LANES][2 * C + 4];
  const int q = threadIdx.x % Q, ln = threadIdx.x / Q;
  float mu[4], rs[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    mu[j] = __ldg(mean + q * 4 + j);
    rs[j] = __ldg(rstd + q * 4 + j);
  }
  float s[4] = {0.f, 0.f, 0.f, 0.f}, sx[4] = {0.f, 0.f, 0.f, 0.f};
  for (long long px = (long long)blockIdx.x * LANES + ln; px < P; px += (long long)gridDim.x * LANES) {
    const uint2 gd = *reinterpret_cast<const uint2*>(dy + px * C + q * 4);
    const uint2 xu = *reinterpret_cast<const uint2*>(xr + px * C + q * 4);
    float g[4] = {bf_lo(gd.x), bf_hi(gd.x), bf_lo(gd.y), bf_hi(gd.y)};
    if (dp.p > 0.f) {
      const float4 k = cv_keep4(dp, (unsigned long long)px * Q + q);
      g[0] *= k.x; g[1] *= k.y; g[2] *= k.z; g[3] *= k.w;
    }
    const float2 a = h2_to_f2(xu.x), b = h2_to_f2(xu.y);
    const float xv[4] = {a.x, a.y, b.x, b.y};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      s[j] += g[j];
      sx[j] = fmaf(g[j], (xv[j] - mu[j]) * rs[j], sx[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    red[ln][q * 4 + j] = s[j];
    red[ln][C + q * 4 + j] = sx[j];
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * C; i += 256) {
    float t = 0.f;
    for (int l = 0; l < LANES; ++l) t += red[l][i];
    partial[(size_t)blockIdx.x * 2 * C + i] = t;
  }
}

// dz = (xr > 0) * gamma * rstd * (g - [batch] (mean_g + xhat * mean_gx)),  g = dy o keep.
// sums [2, C] = (sum g | sum g xhat) over all P pixels; batch_stats == 0: running statistics (eval): the
// correction terms vanish.
__global__ void __launch_bounds__(256)
    bn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ dy, const __half* __restrict__ xr,
                        const float* __restrict__ gamma, const float* __restrict__ mean,
                        const float* __restrict__ rstd, const float* __restrict__ sums, int batch_stats,
                        __nv_bfloat16* __restrict__ dz, long long P, int C, ConvDropout dp) {
  const int Q = C / 4;
  const long long total = P * Q;
  const float inv_p = 1.0f / (float)P;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c0 = (int)(i % Q) * 4;
    const uint2 gd = *reinterpret_cast<const uint2*>(dy + i * 4);
    const uint2 xu = *reinterpret_cast<const uint2*>(xr + i * 4);
    float g[4] = {bf_lo(gd.x), bf_hi(gd.x), bf_lo(gd.y), bf_hi(gd.y)};
    if (dp.p > 0.f) {
      const float4 k = cv_keep4(dp, (unsigned long long)i);
      g[0] *= k.x; g[1] *= k.y; g[2] *= k.z; g[3] *= k.w;
    }
    const float2 a = h2_to_f2(xu.x), b = h2_to_f2(xu.y);
    const float xv[4] = {a.x, a.y, b.x, b.y};
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = c0 + j;
      const float rs = __ldg(rstd + c);
      float v = g[j];
      if (batch_stats) {
        const float xh = (xv[j] - __ldg(mean + c)) * rs;
        v -= __ldg(sums + c) * inv_p + xh * (__ldg(sums + C + c) * inv_p);
      }
      o[j] = (xv[j] > 0.f) ? v * __ldg(gamma + c) * rs : 0.f;
    }
    *reinterpret_cast<uint2*>(dz + i * 4) = make_uint2(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]));
  }
}

// ------------------------------------------------------------------ conv2 wgrad operand
// colT[(tap*C + ci), pix] = y1[b, 2*t2 + kh - 1, 2*f2 + kw - 1, ci]  (0 outside), bf16, pitch ldt >= P2.
// Block: one tap x 64 output pixels x 64 channels, transposed through shared memory.
__global__ void __launch_bounds__(256)
    im2col_t_kernel(const __half* __restrict__ y1, __nv_bfloat16* __restrict__ colT, long long ldt, int B, int T1,
                    int F1, int T2, int F2, int C) {
  __shared__ __align__(16) __nv_bfloat16 tileT[64][72];  // [ci][pix]
  const long long P2 = (long long)B * T2 * F2;
  const long long p0 = (long long)blockIdx.x * 64;
  const int tap = blockIdx.y % 9, cblk = blockIdx.y / 9;  // 64-channel block
  const int kh = tap / 3, kw = tap - kh * 3;
  const int tx = threadIdx.x & 7, ty = threadIdx.x >> 3;  // 8 channel octets x 32 pixels, 2 passes
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    const int pl = ty + pass * 32;
    const long long pix = p0 + pl;
    uint4 u = make_uint4(0, 0, 0, 0);
    if (pix < P2) {
      const int f2 = (int)(pix % F2);
      const long long r = pix / F2;
      const int t2 = (int)(r % T2), b = (int)(r / T2);
      const int t1 = 2 * t2 + kh - 1, f1 = 2 * f2 + kw - 1;
      if (t1 >= 0 && t1 < T1 && f1 >= 0 && f1 < F1)
        u = *reinterpret_cast<const uint4*>(y1 + (((long long)b * T1 + t1) * F1 + f1) * C + cblk * 64 + tx * 8);
    }
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = h2_to_f2(w[j]);
      tileT[tx * 8 + 2 * j][pl] = __float2bfloat16_rn(f.x);
      tileT[tx * 8 + 2 * j + 1][pl] = __float2bfloat16_rn(f.y);
    }
  }
  __syncthreads();
  const int ci = threadIdx.x >> 2, seg = (threadIdx.x & 3) * 16;
  __nv_bfloat16* op = colT + ((long long)tap * C + cblk * 64 + ci) * ldt + p0 + seg;
  if (p0 + seg + 15 < P2 && (ldt & 7) == 0) {
    const uint4* sp = reinterpret_cast<const uint4*>(&tileT[ci][seg]);
    reinterpret_cast<uint4*>(op)[0] = sp[0];
    reinterpret_cast<uint4*>(op)[1] = sp[1];
  } else {
    for (int j = 0; j < 16; ++j)
      if (p0 + seg + j < P2) op[j] = tileT[ci][seg + j];
  }
}

// conv2 dgrad, second half: dy1[b, t1, f1, ci] = sum over taps (kh, kw) with t1 = 2*t2 + kh - 1, f1 = 2*f2 + kw - 1
// of dcol[pix(b, t2, f2), tap*C + ci]   (dcol [P2, 9C] bf16 = dz2 @ W2 from the tcgen05 GEMM).  8 channels / thread.
__global__ void __launch_bounds__(256)
    col2im_kernel(const __nv_bfloat16* __restrict__ dcol, __nv_bfloat16* __restrict__ dy1, int B, int T1, int F1,
                  int T2, int F2, int C) {
  const int oct = C / 8;
  const long long total = (long long)B * T1 * F1 * oct;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c0 = (int)(i % oct) * 8;
    long long r = i / oct;
    const int f1 = (int)(r % F1);
    r /= F1;
    const int t1 = (int)(r % T1), b = (int)(r / T1);
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int tt = t1 + 1 - kh;
      if (tt < 0 || (tt & 1) || (tt >> 1) >= T2) continue;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int ff = f1 + 1 - kw;
        if (ff < 0 || (ff & 1) || (ff >> 1) >= F2) continue;
        const long long pix = ((long long)b * T2 + (tt >> 1)) * F2 + (ff >> 1);
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(dcol + pix * 9 * C + (kh * 3 + kw) * C + c0));
        acc[0] += bf_lo(u.x); acc[1] += bf_hi(u.x); acc[2] += bf_lo(u.y); acc[3] += bf_hi(u.y);
        acc[4] += bf_lo(u.z); acc[5] += bf_hi(u.z); acc[6] += bf_lo(u.w); acc[7] += bf_hi(u.w);
      }
    }
    *reinterpret_cast<uint4*>(dy1 + i * 8) =
        make_uint4(pack_bf16x2(acc[0], acc[1]), pack_bf16x2(acc[2], acc[3]), pack_bf16x2(acc[4], acc[5]),
                   pack_bf16x2(acc[6], acc[7]));
  }
}

// ------------------------------------------------------------------ conv1 weight / bias gradient
// dW1[co, tap] = sum_pix dz1[pix, co] * x[b, 2*t1 + kh - 1, 2*f1 + kw - 1];  db1[co] = sum_pix dz1[pix, co].
// A block walks output rows (b, t1): the three input rows a row of outputs touches are staged once in shared
// memory with their zero halo (every one of the C channel threads of a pixel reads the same nine values, as
// broadcasts), thread <-> (channel, pixel lane) accumulates its 9 + 1 sums in registers over all its rows, and
// the block leaves one partial [C, 10] (9 taps | bias).  (The first version recomputed the pixel -> (b, t1, f1)
// index arithmetic and nine predicated global loads per element: 489 us at cfg2 against a 20 us HBM floor.)
template <int C>
__global__ void __launch_bounds__(256)
    conv1_wgrad_kernel(const __nv_bfloat16* __restrict__ dz1, const float* __restrict__ x, int B, int T, int F,
                       int T1, int F1, float* __restrict__ partial) {
  constexpr int LANES = 256 / C;
  extern __shared__ float cw_smem[];
  float* xs = cw_smem;                 // [3][F + 2]: input rows 2*t1-1 .. 2*t1+1, columns -1 .. F
  float* red = cw_smem + 3 * (F + 2);  // [LANES][C * 10]
  const int co = threadIdx.x % C, ln = threadIdx.x / C;
  const int W = F + 2;
  float acc[10];
#pragma unroll
  for (int k = 0; k < 10; ++k) acc[k] = 0.f;
  const int rows = B * T1;
  for (int row = blockIdx.x; row < rows; row += gridDim.x) {
    const int t1 = row % T1, b = row / T1;
    __syncthreads();  // the previous row's values have been consumed
    for (int i = threadIdx.x; i < 3 * W; i += 256) {
      const int kh = i / W, c = i - kh * W - 1;  // input column c in [-1, F]
      const int t = 2 * t1 + kh - 1;
      xs[i] = (t >= 0 && t < T && c >= 0 && c < F) ? __ldg(x + ((long long)b * T + t) * F + c) : 0.f;
    }
    __syncthreads();
    const __nv_bfloat16* gp = dz1 + (long long)row * F1 * C + co;
    for (int f1 = ln; f1 < F1; f1 += LANES) {
      const float g = __bfloat162float(gp[(long long)f1 * C]);
      const float* p0 = xs + 2 * f1;  // column 2*f1 - 1 of row kh sits at xs[kh*W + 2*f1]
#pragma unroll
      for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) acc[kh * 3 + kw] = fmaf(g, p0[kh * W + kw], acc[kh * 3 + kw]);
      }
      acc[9] += g;
    }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 10; ++k) red[ln * C * 10 + co * 10 + k] = acc[k];
  __syncthreads();
  for (int i = threadIdx.x; i < C * 10; i += 256) {
    float t = 0.f;
    for (int l = 0; l < LANES; ++l) t += red[l * C * 10 + i];
    partial[(size_t)blockIdx.x * C * 10 + i] = t;
  }
}

// ------------------------------------------------------------------ conv1 data gradient (input features)
// dx[b, t, f] = sum_{kt, kf, c} w1[c, 3kt+kf] dz1[b, (t+1-kt)/2, (f+1-kf)/2, c] over the taps whose indices are
// even and in range (stride 2, padding 1).  Input pixels come in 2x2 blocks (2i..2i+1, 2j..2j+1), one block per
// conv1 output pixel (i, j); a block reads the four dz1 pixels (i|i+1, j|j+1) and every tap of every output lands
// on one of them:
//   dx[2i,   2j  ] = w4 z(i,j)
//   dx[2i,   2j+1] = w3 z(i,j+1) + w5 z(i,j)
//   dx[2i+1, 2j  ] = w1 z(i+1,j) + w7 z(i,j)
//   dx[2i+1, 2j+1] = w0 z(i+1,j+1) + w2 z(i+1,j) + w6 z(i,j+1) + w8 z(i,j)
// A group of C/8 lanes shares a block: lane k owns channels 8k..8k+7 (one 16-byte load per dz1 pixel, so a group
// reads each pixel's C channels as one contiguous segment) and keeps those channels' 9 taps in registers for the
// whole grid-stride loop.  The group's four partial sums are combined with a fixed xor butterfly: no atomics, the
// same bits on every call.
template <int C>
__global__ void __launch_bounds__(256)
    conv1_dgrad_kernel(const __nv_bfloat16* __restrict__ dz1, const float* __restrict__ w1, float* __restrict__ dx,
                       int B, int T, int F, int T1, int F1) {
  constexpr int G = C / 8;  // lanes per block: 8 or 16
  const int k = threadIdx.x % G;
  float w[9][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) w[tap][j] = __ldg(w1 + (k * 8 + j) * 9 + tap);
  }
  // the loop runs warp by warp (the butterfly needs every lane): a group past the last block computes zeros.
  // 32-bit indices (the host checks B*T1*F1 < 2^31): 64-bit divisions dominated the first version's time.
  constexpr int GPW = 32 / G;  // groups per warp
  const unsigned blocks = (unsigned)B * T1 * F1;
  const unsigned stride = gridDim.x * (blockDim.x / 32) * GPW;
  for (unsigned base = (blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32) * GPW; base < blocks; base += stride) {
    const unsigned blk = base + (threadIdx.x % 32) / G;
    const bool valid = blk < blocks;
    const unsigned r = blk / F1;
    const int j = (int)(blk - r * F1), i = (int)(r % T1), b = (int)(r / T1);
    const bool right = valid && j + 1 < F1, down = valid && i + 1 < T1;
    const __nv_bfloat16* p = dz1 + (size_t)blk * C + k * 8;
    const uint4 zero = make_uint4(0, 0, 0, 0);
    const uint4 u00 = valid ? __ldg(reinterpret_cast<const uint4*>(p)) : zero;
    const uint4 u01 = right ? __ldg(reinterpret_cast<const uint4*>(p + C)) : zero;
    const uint4 u10 = down ? __ldg(reinterpret_cast<const uint4*>(p + (size_t)F1 * C)) : zero;
    const uint4 u11 = right && down ? __ldg(reinterpret_cast<const uint4*>(p + (size_t)(F1 + 1) * C)) : zero;
    const uint32_t a00[4] = {u00.x, u00.y, u00.z, u00.w}, a01[4] = {u01.x, u01.y, u01.z, u01.w};
    const uint32_t a10[4] = {u10.x, u10.y, u10.z, u10.w}, a11[4] = {u11.x, u11.y, u11.z, u11.w};
    // one accumulator per tap: nine independent FMA chains of 8 instead of one chain of 32 for dx[2i+1, 2j+1]
    float acc[9];
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) acc[tap] = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int h = q >> 1;
      const float z00 = (q & 1) ? bf_hi(a00[h]) : bf_lo(a00[h]), z01 = (q & 1) ? bf_hi(a01[h]) : bf_lo(a01[h]);
      const float z10 = (q & 1) ? bf_hi(a10[h]) : bf_lo(a10[h]), z11 = (q & 1) ? bf_hi(a11[h]) : bf_lo(a11[h]);
      acc[4] = fmaf(w[4][q], z00, acc[4]);
      acc[3] = fmaf(w[3][q], z01, acc[3]);
      acc[5] = fmaf(w[5][q], z00, acc[5]);
      acc[1] = fmaf(w[1][q], z10, acc[1]);
      acc[7] = fmaf(w[7][q], z00, acc[7]);
      acc[0] = fmaf(w[0][q], z11, acc[0]);
      acc[2] = fmaf(w[2][q], z10, acc[2]);
      acc[6] = fmaf(w[6][q], z01, acc[6]);
      acc[8] = fmaf(w[8][q], z00, acc[8]);
    }
    float s00 = acc[4], s01 = acc[3] + acc[5], s10 = acc[1] + acc[7], s11 = (acc[0] + acc[2]) + (acc[6] + acc[8]);
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) {
      s00 += __shfl_xor_sync(0xffffffffu, s00, o);
      s01 += __shfl_xor_sync(0xffffffffu, s01, o);
      s10 += __shfl_xor_sync(0xffffffffu, s10, o);
      s11 += __shfl_xor_sync(0xffffffffu, s11, o);
    }
    // lanes 0..3 of the group store the four outputs that exist (T and F may be odd)
    if (valid && k < 4) {
      const int dt = k >> 1, df = k & 1;
      const int t = 2 * i + dt, f = 2 * j + df;
      if (t < T && f < F) {
        const float v = k == 0 ? s00 : k == 1 ? s01 : k == 2 ? s10 : s11;
        dx[((size_t)b * T + t) * F + f] = v;
      }
    }
  }
}

static inline int cv_grid(long long n, int cap_mult) {
  long long g = (n + 255) / 256;
  const long long cap = (long long)num_sms() * cap_mult;
  if (g > cap) g = cap;
  return (int)(g < 1 ? 1 : g);
}

}  // namespace fbkst

using namespace fbkst;

extern "C" int fbkst_bn_partial_blocks(void) { return num_sms() * 4; }

/* partial: [fbkst_bn_partial_blocks(), 2, C] floats */
extern "C" int fbkst_bn_batch_stats(const void* y_f16, int64_t pixels, int C, const float* gamma, const float* beta,
                                    float eps, float momentum, float* running_mean, float* running_var,
                                    float* mean, float* rstd, float* scale, float* shift, float* partial,
                                    fbkst_stream_t stream) {
  FBKST_REQUIRE(y_f16 && gamma && beta && mean && rstd && scale && shift && partial && pixels > 0,
                "fbkst_bn_batch_stats: bad arguments");
  FBKST_REQUIRE(C == 64 || C == 128, "fbkst_bn_batch_stats: C must be 64 or 128");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int G = fbkst_bn_partial_blocks();
  if (C == 64)
    bn_stats_kernel<64><<<G, 256, 0, st>>>(reinterpret_cast<const __half*>(y_f16), pixels, partial);
  else
    bn_stats_kernel<128><<<G, 256, 0, st>>>(reinterpret_cast<const __half*>(y_f16), pixels, partial);
  FBKST_CHECK_CUDA(cudaGetLastError());
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(partial, G, C, (double)pixels, gamma, beta, eps, momentum,
                                                      running_mean, running_var, mean, rstd, scale, shift);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_bn_apply(const void* x_f16, void* y_f16, const float* scale, const float* shift,
                              int64_t pixels, int C, float p, uint64_t seed, int site, fbkst_stream_t stream) {
  FBKST_REQUIRE(x_f16 && y_f16 && scale && shift && pixels > 0 && C % 8 == 0, "fbkst_bn_apply: bad arguments");
  FBKST_REQUIRE(p >= 0.f && p < 1.f, "fbkst_bn_apply: p must be in [0, 1)");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  bn_apply_kernel<<<cv_grid(pixels * (C / 8), 8), 256, 0, st>>>(reinterpret_cast<const __half*>(x_f16),
                                                               reinterpret_cast<__half*>(y_f16), scale, shift,
                                                               pixels, C, cv_make_dropout(p, seed, site));
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

/* dz [P, C] bf16 = autograd of dropout(BatchNorm(relu_out)) . relu w.r.t. the conv output, given dy [P, C] bf16;
 * sums [2, C] receives (dbeta | dgamma);  partial: [fbkst_bn_partial_blocks(), 2, C] floats.  With running
 * statistics dz does not read the sums: sums == NULL (and partial == NULL) skips their reduction pass. */
extern "C" int fbkst_bn_relu_bwd(const void* dy_bf16, const void* relu_out_f16, const float* gamma,
                                 const float* mean, const float* rstd, int batch_stats, void* dz_bf16,
                                 float* sums, float* partial, int64_t pixels, int C, float p, uint64_t seed,
                                 int site, fbkst_stream_t stream) {
  FBKST_REQUIRE(dy_bf16 && relu_out_f16 && gamma && mean && rstd && dz_bf16 && pixels > 0,
                "fbkst_bn_relu_bwd: bad arguments");
  FBKST_REQUIRE(sums ? partial != nullptr : !batch_stats,
                "fbkst_bn_relu_bwd: sums and partial are required (batch statistics read the sums)");
  FBKST_REQUIRE(C == 64 || C == 128, "fbkst_bn_relu_bwd: C must be 64 or 128");
  FBKST_REQUIRE(p >= 0.f && p < 1.f, "fbkst_bn_relu_bwd: p must be in [0, 1)");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const ConvDropout dp = cv_make_dropout(p, seed, site);
  const int G = fbkst_bn_partial_blocks();
  const __nv_bfloat16* dy = reinterpret_cast<const __nv_bfloat16*>(dy_bf16);
  const __half* xr = reinterpret_cast<const __half*>(relu_out_f16);
  if (sums != nullptr) {
    if (C == 64)
      bn_bwd_reduce_kernel<64><<<G, 256, 0, st>>>(dy, xr, mean, rstd, pixels, partial, dp);
    else
      bn_bwd_reduce_kernel<128><<<G, 256, 0, st>>>(dy, xr, mean, rstd, pixels, partial, dp);
    FBKST_CHECK_CUDA(cudaGetLastError());
    int rc = fbkst_reduce_sum(partial, G, 2 * C, 1, 2 * C, 2 * C, sums, 2 * C, 1.0f, stream);
    if (rc) return rc;
  }
  bn_bwd_apply_kernel<<<cv_grid(pixels * (C / 4), 8), 256, 0, st>>>(dy, xr, gamma, mean, rstd, sums, batch_stats,
                                                                   reinterpret_cast<__nv_bfloat16*>(dz_bf16),
                                                                   pixels, C, dp);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_conv2_im2col_t(const void* y1_f16, void* colT_bf16, int64_t ldt, int B, int T1, int F1, int C,
                                    fbkst_stream_t stream) {
  FBKST_REQUIRE(y1_f16 && colT_bf16 && B > 0 && T1 > 0 && F1 > 0 && (C == 64 || C == 128),
                "fbkst_conv2_im2col_t: bad arguments");
  const int T2 = (T1 + 1) / 2, F2 = (F1 + 1) / 2;
  const long long P2 = (long long)B * T2 * F2;
  FBKST_REQUIRE(ldt >= P2, "fbkst_conv2_im2col_t: pitch smaller than the pixel count");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  dim3 grid((unsigned)((P2 + 63) / 64), 9 * (C / 64));
  im2col_t_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const __half*>(y1_f16),
                                        reinterpret_cast<__nv_bfloat16*>(colT_bf16), ldt, B, T1, F1, T2, F2, C);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

extern "C" int fbkst_conv2_col2im(const void* dcol_bf16, void* dy1_bf16, int B, int T1, int F1, int C,
                                  fbkst_stream_t stream) {
  FBKST_REQUIRE(dcol_bf16 && dy1_bf16 && B > 0 && T1 > 0 && F1 > 0 && C % 8 == 0, "fbkst_conv2_col2im: bad arguments");
  const int T2 = (T1 + 1) / 2, F2 = (F1 + 1) / 2;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  col2im_kernel<<<cv_grid((long long)B * T1 * F1 * (C / 8), 8), 256, 0, st>>>(
      reinterpret_cast<const __nv_bfloat16*>(dcol_bf16), reinterpret_cast<__nv_bfloat16*>(dy1_bf16), B, T1, F1, T2,
      F2, C);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}

/* dw1b [C, 10] fp32 = (dW1[co, 0..8] | db1[co]);  partial: [fbkst_bn_partial_blocks(), C, 10] floats */
extern "C" int fbkst_conv1_wgrad(const void* dz1_bf16, const float* x, float* dw1b, float* partial, int B, int T,
                                 int F, int C, fbkst_stream_t stream) {
  FBKST_REQUIRE(dz1_bf16 && x && dw1b && partial && B > 0 && T > 0 && F > 0 && (C == 64 || C == 128),
                "fbkst_conv1_wgrad: bad arguments");
  const int T1 = (T + 1) / 2, F1 = (F + 1) / 2;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int G = fbkst_bn_partial_blocks();
  const __nv_bfloat16* dz = reinterpret_cast<const __nv_bfloat16*>(dz1_bf16);
  const size_t smem = sizeof(float) * (3 * (size_t)(F + 2) + (size_t)(256 / C) * C * 10);
  FBKST_REQUIRE(smem <= 48 * 1024, "fbkst_conv1_wgrad: F=%d too wide for the staging buffer", F);
  if (C == 64)
    conv1_wgrad_kernel<64><<<G, 256, smem, st>>>(dz, x, B, T, F, T1, F1, partial);
  else
    conv1_wgrad_kernel<128><<<G, 256, smem, st>>>(dz, x, B, T, F, T1, F1, partial);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return fbkst_reduce_sum(partial, G, (int64_t)C * 10, 1, C * 10, C * 10, dw1b, C * 10, 1.0f, stream);
}

/* dx [B,T,F] fp32 = gradient of conv1's input from dz1 [B,T1,F1,C] bf16 and w1 [C, 9] fp32 (every input position,
 * padded frames included) */
extern "C" int fbkst_conv1_dgrad(const void* dz1_bf16, const float* w1, float* dx, int B, int T, int F, int C,
                                 fbkst_stream_t stream) {
  FBKST_REQUIRE(dz1_bf16 && w1 && dx && B > 0 && T > 0 && F > 0 && (C == 64 || C == 128),
                "fbkst_conv1_dgrad: bad arguments");
  const int T1 = (T + 1) / 2, F1 = (F + 1) / 2;
  FBKST_REQUIRE((long long)B * T1 * F1 < (1LL << 31) - 256 * 32, "fbkst_conv1_dgrad: batch too large");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const long long lanes = (long long)B * T1 * F1 * (C / 8);
  const __nv_bfloat16* dz = reinterpret_cast<const __nv_bfloat16*>(dz1_bf16);
  if (C == 64)
    conv1_dgrad_kernel<64><<<cv_grid(lanes, 2), 256, 0, st>>>(dz, w1, dx, B, T, F, T1, F1);
  else
    conv1_dgrad_kernel<128><<<cv_grid(lanes, 2), 256, 0, st>>>(dz, w1, dx, B, T, F, T1, F1);
  FBKST_CHECK_CUDA(cudaGetLastError());
  return FBKST_OK;
}
