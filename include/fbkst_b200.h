/*
 * fbkst_b200 -- C ABI of the B200-native (sm_100a) speech-translation encoder hot path.
 *
 * Drop-in boundary for the forward of FBK-fairseq-ST's ConvolutionalTransformerEncoder
 * (reference: examples/speech_recognition/models/conv_transformer.py:195-291 and the
 * modules it calls).  The reference has no native code on this path (every op is a
 * PyTorch call), so each entry point below names the reference *Python* call site it
 * replaces; INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless named h_*;
 *   - every function launches on `stream` and returns immediately (no host sync unless stated);
 *   - return 0 on success, a negative FBKST_ERR_* otherwise; fbkst_last_error() returns the
 *     message of the last failure on the calling thread.  Allocation failures contain the
 *     substring "out of memory" (fairseq/trainer.py:394-405 greps for it);
 *   - the library never allocates device memory for results: callers own every buffer;
 *   - time-major activations: row m = t * B + b  (the reference's T x B x C layout);
 *   - bf16 = __nv_bfloat16 storage, fp32 accumulation everywhere.
 */
#ifndef FBKST_B200_H_
#define FBKST_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* fbkst_stream_t;

enum {
  FBKST_OK = 0,
  FBKST_ERR_ARG = -1,  /* bad argument / unsupported shape */
  FBKST_ERR_CUDA = -2, /* CUDA runtime / driver error */
  FBKST_ERR_OOM = -3   /* CUDA out of memory */
};

enum { FBKST_BF16 = 0, FBKST_F32 = 1 };

enum { FBKST_CTC_AVG = 0, FBKST_CTC_WEIGHTED = 1, FBKST_CTC_SOFTMAX = 2 };

/* query modes of fbkst_dec_self_attn_fwd */
enum { FBKST_SA_INCREMENTAL = 0, FBKST_SA_FULL = 1, FBKST_SA_CAUSAL = 2 };

/* epilogue flags of fbkst_linear_bf16 */
enum {
  FBKST_EPI_RELU = 1,      /* y = max(y, 0) after the bias                                  */
  FBKST_EPI_OUT_F32 = 2,   /* out is fp32 (default bf16)                                    */
  FBKST_EPI_AB_F16 = 16    /* A and W hold IEEE fp16 instead of bf16 (the conv front end)    */
};

const char* fbkst_last_error(void);
int fbkst_abi_version(void);
/* 1 when a CUDA device of compute capability 10.x is present, else 0 (never a CPU fallback) */
int fbkst_device_ok(void);

/* ---- a1: per-utterance fbank mean/variance normalisation ------------------------------
 * replaces examples/speech_recognition/data/data_utils.py:9-24 (apply_mv_norm), called at
 * data/fbank_dataset.py:44-45.  x, y: [B, T, F] fp32 (y may alias x); lengths[B] int32.
 * Rows t >= lengths[b] are written as 0.  workspace: B*F*2 doubles. */
int fbkst_cmvn_f32(const float* x, float* y, const int32_t* lengths, int B, int T, int F,
                   double* workspace, fbkst_stream_t stream);

/* ---- next row N2: collate (+ optional CMVN) on device ---------------------------------------
 * replaces examples/speech_recognition/data/collaters.py:43-56 (_collate_frames: zero-padded
 * B x T x F batch) for features that arrive RAGGED: packed [sum(lengths), F] fp32 holds the
 * utterances back to back, starts[b] (int64) is the first frame of the utterance that goes to
 * batch slot b (the host has already sorted slots by descending length, collaters.py:89-92),
 * lengths[b] its frame count.  out [B, T, F] fp32, rows t >= lengths[b] are 0.  normalize != 0
 * additionally applies apply_mv_norm per utterance (data/data_utils.py:9-24) in the same pass;
 * workspace: B*F*2 doubles (may be NULL when normalize == 0). */
int fbkst_collate_cmvn_f32(const float* packed, const int64_t* starts, const int32_t* lengths,
                           float* out, int B, int T, int F, int normalize, double* workspace,
                           fbkst_stream_t stream);

/* ---- a2 (conv 1): Conv2d(1->C,k3,s2,p1)+bias -> ReLU -> BatchNorm(eval affine) -----------
 * replaces conv_transformer.py:203-214 for i=0.  x [B,T,F] fp32; w [C,9] fp32; bias,
 * bn_scale, bn_shift [C] fp32 (scale = gamma/sqrt(var+eps), shift = beta - mean*scale);
 * y [B,T1,F1,C] IEEE fp16 channels-last (saturating conversion), T1=ceil(T/2), F1=ceil(F/2).  C must
 * be 64 or 128.  The conv front end (conv1, conv2, fc3 operands) runs in fp16, not bf16: its six
 * operand roundings in series otherwise dominate the encoder's output error (DESIGN.md section 4). */
int fbkst_conv1_relu_bn(const float* x, const float* w, const float* bias, const float* bn_scale,
                        const float* bn_shift, void* y, int B, int T, int F, int C,
                        fbkst_stream_t stream);

/* ---- a2 (conv 2): Conv2d(C->C,k3,s2,p1)+bias -> ReLU -> BatchNorm(eval affine) -----------
 * replaces conv_transformer.py:203-214 for i=1 as a TMA-fed implicit GEMM on tcgen05.
 * x [B,T1,F1,C] fp16 channels-last; w_taps [9][C][C] fp16 (tap = kh*3+kw, then out-ch,
 * in-ch); y [B,T2,F2,C] fp16 channels-last (T2=ceil(T1/2), F2=ceil(F1/2)), i.e. row
 * (b,t) of the fc3 operand with the flatten order (f, c). */
int fbkst_conv2_relu_bn(const void* x, const void* w_taps, const float* bias,
                        const float* bn_scale, const float* bn_shift, void* y, int B, int T1,
                        int F1, int C, fbkst_stream_t stream);

/* ---- generic fused linear: out = epi(A @ W^T) on tcgen05 --------------------------------
 * replaces every F.linear / nn.Linear on the path (conv_transformer.py:227,279;
 * local_attention.py:178,141; fairseq/modules/transformer_layer.py:131-133).
 * A [M,K] bf16 (row pitch lda), W [N,K] bf16 (row pitch ldw), bias [N] fp32 or NULL.
 * y = A W^T + bias; ReLU if FBKST_EPI_RELU; then, if residual != NULL (requires FBKST_EPI_OUT_F32):
 *   y += residual[m, n]   (fp32, row pitch ldr)
 * out row m, out pitch ldo; dtype by flag.
 * m_limit (device, may be NULL): only rows m < m_limit[0] * m_limit_mult are computed -- the
 * number of rows that are valid after CTC compression is known only on the device, so the
 * layers after it are launched for the worst case and skip the tiles beyond the limit
 * (no host synchronisation in the middle of the forward).
 * K % 8 == 0; lda, ldw % 8 == 0; all bases 16-byte aligned. */
int fbkst_linear_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                      const float* residual, int64_t ldr, void* out, int64_t ldo, int M, int N,
                      int K, int flags, const int32_t* m_limit, int m_limit_mult, fbkst_stream_t stream);

/* ---- a6/a8 fused: linear with the pre-LayerNorm of the reference's residual block folded in ---
 * replaces the pairs  LayerNorm -> F.linear  of fairseq/modules/transformer_layer.py:108-110
 * (self_attn_layer_norm -> in-projection, local_attention.py:178) and :126-131 (final_layer_norm
 * -> fc1) without a LayerNorm kernel, using
 *     LN(x) W^T + b = rstd(x) * (x W''^T) + c,
 *     W''[n,k] = gamma[k] W[n,k] - mean_k(gamma[k] W[n,k]),   c[n] = b[n] + sum_k beta[k] W[n,k]
 * (every row of W'' sums to zero, so the row mean of x drops out; W'' and c are prepared by the host).
 * Same operands and flags as fbkst_linear_bf16, plus
 *   producer side (residual epilogue, i.e. out_proj / fc2):  out_bf16 [M,N] bf16 (pitch ldob)
 *     receives bf16(out) and row_stats_out [M, ceil(N/128)] x 2 fp32 the (mean, M2) of each
 *     128-column slice of every output row; both NULL to skip.  N % 32 == 0;
 *   consumer side (plain epilogue, i.e. QKV / fc1 fed with out_bf16 as A and W'' as W):
 *     row_stats_in [M, ceil(K/128)] x 2 fp32 as written by the producer (K == LayerNorm width);
 *     the epilogue computes y = rstd * acc + bias with rstd = 1/sqrt(var + ln_eps); NULL: rstd = 1. */
int fbkst_linear_ln_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias,
                         const float* residual, int64_t ldr, void* out, int64_t ldo, int M, int N,
                         int K, int flags, const float* row_stats_in, float ln_eps, void* out_bf16,
                         int64_t ldob, float* row_stats_out, const int32_t* m_limit,
                         int m_limit_mult, fbkst_stream_t stream);

/* Row statistics + bf16 copy of an x that does not come out of a residual GEMM (fc3 output,
 * CTC-compressed rows): xb = bf16(x), row_stats [M, D/128] x 2 fp32 as above.  Same D as
 * fbkst_layernorm; m_limit as in fbkst_linear_bf16. */
int fbkst_row_stats_cast(const float* x, void* xb, float* row_stats, int M, int D,
                         const int32_t* m_limit, int m_limit_mult, fbkst_stream_t stream);

/* ---- a3/a4 tail: conv_transformer.py:225-229 (transpose(0,1) of the fc3 output + positions) fused with
 * the first layer's row statistics.  src [B*L, D] fp32 in (b, t) row order (the fc3 GEMM output) ->
 * x [L*B, D] fp32 time-major (row t*B + b), x += table[t+1] inside the utterance / table[0] (the
 * padding row) beyond lengths[b] when table != NULL, xb = bf16(x), row_stats as fbkst_row_stats_cast. */
int fbkst_embed_remap_stats(const float* src, const float* table, int64_t ld_table,
                            const int32_t* lengths, float* x, void* xb, float* row_stats, int L, int B,
                            int D, fbkst_stream_t stream);

/* ---- a8: LayerNorm over the last dim (eps 1e-5, affine) ----------------------------------
 * replaces fairseq/modules/layer_norm.py:29-32 call sites (transformer_layer.py:108,126;
 * conv_transformer.py:253-254).  x [M,D] fp32 -> y [M,D] bf16 or fp32.  D in {128,256,384,512,
 * 768,1024}.  m_limit as in fbkst_linear_bf16. */
int fbkst_layernorm(const float* x, const float* gamma, const float* beta, void* y, int out_dtype,
                    int M, int D, float eps, const int32_t* m_limit, int m_limit_mult,
                    fbkst_stream_t stream);

/* ---- a7: self-attention core with key-padding mask and log distance penalty --------------
 * replaces local_attention.py:115-139 (and the math of F.multi_head_attention_forward when
 * log_penalty = 0).  qkv [L*B, 3D] bf16, row m = t*B+b, columns [q | k | v], q pre-scaled by
 * head_dim^-0.5 (folded into the projection weights); heads of 64 channels.
 * out [L*B, D] bf16.  lengths[B] int32: keys t >= lengths[b] are masked; query rows in tiles
 * entirely beyond lengths[b] are written as 0.  scores - ln(max(1,|i-j|)) if log_penalty. */
int fbkst_attention_fwd(const void* qkv, void* out, const int32_t* lengths, int L, int B, int H,
                        int log_penalty, fbkst_stream_t stream);
/* Same, for a caller that only consumes query rows t < *q_limit (device int32, e.g. the maximum length
 * after CTC compression, known only on the device): query tiles that start at or beyond *q_limit AND
 * lie entirely beyond lengths[b] are left untouched instead of being zero-filled. */
int fbkst_attention_fwd_limited(const void* qkv, void* out, const int32_t* lengths, int L, int B, int H,
                                int log_penalty, const int32_t* q_limit, fbkst_stream_t stream);

/* ---- F: fp32-accurate inference path (encoder.precision = "fp32"), split-TF32 tensor-core kernels -------
 * Every operand x is split in shared memory into hi = tf32(x) (rounded) and lo = tf32(x - hi); products are
 * hi.hi + hi.lo + lo.hi in one fp32 accumulator (about 21 significant bits per operand; fp32 in HBM).
 *
 * Linear: replaces every F.linear / nn.Linear on the fp32 path (conv_transformer.py:227,279;
 * local_attention.py:178,141; transformer_layer.py:131-133) and conv2 over fbkst_conv2_im2col_f32
 * (conv_transformer.py:205-212).  A [M,K] fp32 (pitch lda), W [N,K] fp32 (pitch ldw), K, lda, ldw % 4 == 0.
 * y = A W^T + bias; ReLU if relu; y = y * col_scale[n] + col_shift[n] if col_scale (eval BatchNorm after the
 * ReLU); y += residual[m, n] (pitch ldr) if residual.  out [M, N] fp32 (pitch ldo).  m_limit (device int32 [1]
 * or NULL): only rows m < *m_limit * m_limit_mult are computed (the layers after CTC compression). */
int fbkst_linear_tf32x3(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
                        const float* col_scale, const float* col_shift, const float* residual, int64_t ldr,
                        float* out, int64_t ldo, int M, int N, int K, int relu, const int32_t* m_limit,
                        int m_limit_mult, fbkst_stream_t stream);
/* Attention: replaces local_attention.py:115-139 (log_penalty = 1) and the math of
 * F.multi_head_attention_forward (log_penalty = 0) as fbkst_attention_fwd does, in fp32: qkv [L*B, 3D] fp32
 * (q pre-scaled by head_dim^-0.5), out [L*B, D] fp32, H <= 16, fp32 softmax.  Query rows of 128-row tiles
 * entirely beyond lengths[b] are zero; with q_limit (device int32 [1] or NULL) tiles starting at or beyond
 * *q_limit are left untouched. */
int fbkst_attention_tf32x3(const float* qkv, float* out, const int32_t* lengths, int L, int B, int H,
                           int log_penalty, const int32_t* q_limit, fbkst_stream_t stream);
/* conv1 + ReLU + eval BatchNorm in fp32 (conv_transformer.py:205-212, first convolution): x [B,T,F] fp32,
 * w [C,9] fp32 -> y [B,T1,F1,C] fp32 channels-last. */
int fbkst_conv1_relu_bn_f32(const float* x, const float* w, const float* bias, const float* bn_scale,
                            const float* bn_shift, float* y, int B, int T, int F, int C, fbkst_stream_t stream);
/* conv2's patches: y1 [B,T1,F1,C] fp32 -> col [B*T2*F2, 9*C] fp32, column (kt*3 + kf)*C + c, zero padding 1,
 * stride 2.  C % 4 == 0. */
int fbkst_conv2_im2col_f32(const float* y1, float* col, int B, int T1, int F1, int C, fbkst_stream_t stream);

/* ---- a4: sinusoidal position table (row 0 = zeros) ---------------------------------------
 * replaces fairseq/modules/sinusoidal_positional_embedding.py:36-58.  table [rows, D] fp32. */
int fbkst_sinusoidal_table(float* table, int rows, int D, fbkst_stream_t stream);

/* ---- a5: padding mask -----------------------------------------------------------------
 * replaces conv_transformer.py:293-300.  mask [B, L] uint8 (1 = pad); any_pad[1] int32 is
 * set non-zero if some element is padding (the reference returns None otherwise). */
int fbkst_lengths_to_mask(const int32_t* lengths, uint8_t* mask, int32_t* any_pad, int B, int L,
                          fbkst_stream_t stream);

/* ---- a2: length update of the subsampling stack ------------------------------------------
 * replaces `src_lengths = torch.ceil(src_lengths.float() / 2)` per convolution
 * (conv_transformer.py:213).  lengths [B] int64 (lengths_are_i64 != 0, fairseq's dtype) or int32 on the
 * DEVICE -> out [B] int32 = n after `times` halvings (ceil).  Lets the forward accept device-resident
 * lengths (fairseq's utils.move_to_cuda puts them there) without a host round trip. */
int fbkst_subsample_lengths(const void* lengths, int lengths_are_i64, int32_t* out, int B, int times,
                            fbkst_stream_t stream);

/* ---- a9 + a10 step 1 fused: ctc_fc on tcgen05 with the frame arg-max folded into its epilogue --------
 * logits [M, N] fp32 (pitch ldo) = A W^T + bias, exactly as fbkst_linear_bf16 with FBKST_EPI_OUT_F32, and
 * partial [M, ceil(N/128)] x (max, arg-max, sum exp) per 128-column chunk, so that the logits are never re-read
 * (conv_transformer.py:279 + :282-284).  bump_cols [M] int32 (optional): `bump` is added to that column of each
 * row before the store and the arg-max (benchmark / test logit injection, equivalent to a forward hook).
 * (bump >= 0.)  want_sum: also accumulate sum exp and the arg-max column (weighted / softmax pooling need the top
 * probability); without it the epilogue only tracks the chunk maximum.
 * fbkst_ctc_argmax_merge folds the partials: labels [L*B] int32 (-1 for padded frames), top_prob / lse optional;
 * it takes the logits written by the call above (pitch ldv, V columns) to recover the arg-max column inside the
 * row's winning chunk when the partials carry maxima only (128 logits re-read per row). */
int fbkst_linear_argmax_f32(const void* A, int64_t lda, const void* W, int64_t ldw, const float* bias, float* out,
                            int64_t ldo, int M, int N, int K, const int32_t* bump_cols, float bump, int want_sum,
                            float* partial, const int32_t* m_limit, int m_limit_mult, fbkst_stream_t stream);
int fbkst_ctc_argmax_merge(const float* partial, int chunks, const float* logits, int64_t ldv, int V,
                           const int32_t* lengths, int32_t* labels, float* top_prob, float* lse, int L, int B,
                           fbkst_stream_t stream);

/* ---- a10 step 1: CTC argmax (+ probability of the arg-max label) --------------------------
 * replaces conv_transformer.py:282-284 (softmax + per-utterance argmax().tolist()).
 * logits [L*B, ldv] bf16 or fp32 (row m = t*B+b, V valid columns); labels[L*B] int32
 * (-1 for t >= lengths[b]); top_prob[L*B] fp32 = softmax(logits)[label] (0 for padding), or
 * NULL to skip the log-sum-exp (avg strategy).  Ties resolve to the lowest index. */
int fbkst_ctc_argmax(const void* logits, int logits_dtype, int64_t ldv, const int32_t* lengths,
                     int32_t* labels, float* top_prob, int L, int B, int V, fbkst_stream_t stream);

/* Same, plus lse[L*B] fp32 = log(sum_v exp(logits[row, v])) (natural log; 0 for padding rows), or
 * NULL.  log_softmax(logits)[row, v] = logits[row, v] - lse[row]: what the CTC criterion needs
 * (criterions/ctc_multi_loss.py:64-67 log_softmax over the fp32 logits) without materialising
 * the L x B x V log-probabilities. */
int fbkst_ctc_argmax_lse(const void* logits, int logits_dtype, int64_t ldv, const int32_t* lengths,
                         int32_t* labels, float* top_prob, float* lse, int L, int B, int V,
                         fbkst_stream_t stream);

/* ---- a10 step 2 + a11: run-length segmentation and per-frame pooling weights ----------------
 * replaces conv_transformer.py:285-288 (groupby) and :385-426 (CTCCompressStrategy.*).
 * seg_id[L*B] int32: index of the run frame (t,b) belongs to (-1 for padding);
 * seg_start[L*B] int32: seg_start[s*B+b] = first frame of run s of utterance b (s < new length);
 * weight[L*B] fp32: W[b,t,seg_id] (0 for padding); new_lengths[B] int32; max_new_len[1] int32.
 * top_prob may be NULL for FBKST_CTC_AVG. */
int fbkst_ctc_segment(const int32_t* labels, const float* top_prob, const int32_t* lengths,
                      int strategy, int32_t* seg_id, int32_t* seg_start, float* weight,
                      int32_t* new_lengths, int32_t* max_new_len, int L, int B,
                      fbkst_stream_t stream);

/* ---- a10 step 3: segmented weighted reduction (the reference's dense bmm) ------------------
 * replaces conv_transformer.py:290-291.  x [L*B, D] fp32 -> out [L*B, D] fp32 (rows
 * s*B+b; rows with new_lengths[b] <= s < max_new_len + G are written as 0, G = ceil(512/B) + 1
 * guard rows that cover the tile rounding of the row-limited GEMMs run on `out` afterwards; rows
 * beyond are untouched).  seg_id, seg_start, weight as produced by fbkst_ctc_segment.  D % 4 == 0
 * (D % 128 == 0 takes the input-stationary streaming kernel).  Every output row has one writer
 * and a fixed summation order (ascending t): results are run-to-run identical. */
int fbkst_ctc_compress(const float* x, const int32_t* seg_id, const int32_t* seg_start,
                       const float* weight, const int32_t* lengths, const int32_t* new_lengths,
                       const int32_t* max_new_len, float* out, int L, int B, int D,
                       fbkst_stream_t stream);

/* ---- next row N1: the CTC criterion over ctc_out, on device ----------------------------------
 * fbkst_ctc_uer replaces examples/speech_recognition/criterions/CTC_loss.py:31-74
 * (compute_ctc_uer: per-utterance argmax().tolist(), python groupby, blank removal and
 * EditDistance(False).align of utils/wer_utils.py:141-202 with costs match 0 / step 3 / mismatch 4).
 * labels[L*B] int32 as written by fbkst_ctc_argmax on the CTC logits (row t*B+b; frames
 * t >= in_lengths[b] are ignored); targets [B, ldt] int64 (fairseq's padded `target`), the first
 * target_lengths[b] (int32, clamped to Umax) entries of row b are used.
 * errors[B] int32 = number of non-match codes on the alignment path the reference backtracks
 * (same strict-'<' tie-breaks), pred_lengths[B] int32 = tokens left after collapsing,
 * totals[2] int64 = {sum of errors, sum of target lengths} (the reference's batch_errors and
 * batch_total).  Integer work: bit-exact.  Both sequences empty: 0 errors (the reference raises). */
int fbkst_ctc_uer(const int32_t* labels, const int32_t* in_lengths, const int64_t* targets,
                  int64_t ldt, const int32_t* target_lengths, int blank, int32_t* errors,
                  int32_t* pred_lengths, int64_t* totals, int L, int B, int Umax,
                  fbkst_stream_t stream);

/* fbkst_ctc_loss_fwd replaces the F.ctc_loss call of criterions/CTC_loss.py:143-151
 * (reduction="sum", zero_infinity=True) including the log_softmax before it: logits [L*B, ldv]
 * bf16/fp32 (row t*B+b, V valid columns), lse[L*B] from fbkst_ctc_argmax_lse.
 * nll[B] fp32 = -log p(target_b | x_b) (0 where infinite), loss[1] fp32 = their sum in a fixed
 * order.  Forward only (validation / scoring); fp32 log-space alpha recursion. */
int fbkst_ctc_loss_fwd(const void* logits, int logits_dtype, int64_t ldv, const float* lse,
                       const int32_t* in_lengths, const int64_t* targets, int64_t ldt,
                       const int32_t* target_lengths, int blank, float* nll, float* loss, int L,
                       int B, int V, int Umax, fbkst_stream_t stream);

/* ---- next row N3: training-time batch augmentation on device ------------------------------------
 * fbkst_specaugment_f32 replaces examples/speech_recognition/modules/specaugment.py:55-112 (the
 * per-spectrogram slice assignments of `specaugment`, called from tasks/speech_recognition.py:257-258).
 * x [B, T, F] fp32 is masked IN PLACE: bands [B, n_freq + n_time, 2] int32 = (start, width) per
 * utterance, the first n_freq are feature bands (x[b, :, f0:f0+f] = 0), the rest time bands
 * (x[b, t0:t0+t, :] = 0); width 0 = nothing (utterances the `rate` draw skipped).  The host draws
 * the bands with the reference's RNG calls in the reference's order.  Write-only kernel. */
int fbkst_specaugment_f32(float* x, const int32_t* bands, int B, int T, int F, int n_freq, int n_time,
                          fbkst_stream_t stream);

/* fbkst_time_stretch_f32 replaces modules/time_stretch.py:18-57 (TimeStretch.forward +
 * time_stretch_seq: per-window torch.linspace -> round -> long index lists, fancy-indexing per
 * utterance, re-padding on the host and a second H2D).  x [B, T, F] fp32; windows [n_windows, 4] int32
 * = (first, last, count, out_off): the window resamples frames first..last of its utterance to `count`
 * frames written at flat position out_off (= b * T_out + offset) -- the host computes count =
 * int(uniform(low, high) * window_size) with the reference's RNG calls; an utterance the `rate` draw
 * skipped is one window (0, len-1, len, b*T_out).  ids [B, T_out] int32 receives the source frame of
 * every output frame, bit-identical to the reference's index tensors (-1 beyond the new length);
 * out [B, T_out, F] fp32 = x[b, ids[b, j], :] (0 where ids < 0).  16-byte aligned windows. */
int fbkst_time_stretch_f32(const float* x, const int32_t* windows, int n_windows, int32_t* ids,
                           float* out, int B, int T, int T_out, int F, fbkst_stream_t stream);

/* ---- next row N4: decoder cross-attention over the compressed encoder output ---------------------
 * fbkst_xattn_fwd replaces the static_kv path of fairseq/modules/multihead_attention.py:108-367 as the
 * decoder layer calls it (fairseq/modules/transformer_layer.py:339-348) during incremental generation,
 * together with the x beam replication of the encoder output (conv_transformer.py:315-345,
 * fairseq/sequence_generator.py:193-198) and the per-step re-gather of the cached keys/values
 * (multihead_attention.py:407-420): K/V are projected once per UTTERANCE and rows address them through
 * row_map, so replication/reordering never copies K/V.
 *   q        [tgt_len * bsz, D] bf16, row r = t * bsz + b, already scaled by head_dim^-0.5 (:209)
 *   kv       [S, U, 2D] bf16 time-major: columns [0, D) = k_proj(encoder_out), [D, 2D) = v_proj(...)
 *   key_padding_mask [U, S] uint8 (1 = padding key, :330-335) or NULL
 *   row_map  [bsz] int32: utterance (0..U-1) of hypothesis row b; out-of-range -> zero output row
 *   out      [tgt_len * bsz, D] bf16 (heads concatenated; input of out_proj, :353)
 *   attn_w   w_mode 0: unused; 1: [bsz, tgt_len, S] fp32 averaged over heads (:355-362);
 *            2: [H, bsz, tgt_len, S] fp32 per head (need_head_weights)
 *   head_ws  w_mode 1 only: caller-owned scratch [H, bsz, tgt_len, S] fp32 (per-head weights; the
 *            average is taken over it in a fixed order)
 * D = 64 * H, H <= 16; 32 * S + 14.4 KB of shared memory must fit in 200 KB (S <= ~5900). */
int fbkst_xattn_fwd(const void* q, const void* kv, const uint8_t* key_padding_mask,
                    const int32_t* row_map, void* out, float* attn_w, float* head_ws, int w_mode,
                    int S, int U, int bsz, int tgt_len, int H, fbkst_stream_t stream);
/* fbkst_xattn_fwd with fp32 q [tgt_len * bsz, D] (8-byte aligned), kv [S, U, 2D] and out [tgt_len * bsz, D]
 * (16-byte aligned): the fp32-accurate decode path (CrossAttention.precision = "fp32").  Same kernel body,
 * fp32 FMA and softmax; every other argument as above. */
int fbkst_xattn_fwd_f32(const float* q, const float* kv, const uint8_t* key_padding_mask,
                        const int32_t* row_map, float* out, float* attn_w, float* head_ws, int w_mode,
                        int S, int U, int bsz, int tgt_len, int H, fbkst_stream_t stream);

/* ---- next row N5: decoder self-attention over an append-only K/V cache ---------------------------
 * fbkst_dec_self_attn_fwd replaces fairseq/modules/multihead_attention.py:108-367 with
 * self_attention=True as TransformerDecoderLayer.forward calls it (fairseq/modules/transformer_layer.py).  In
 * generation the reference appends each step's key and value to per-hypothesis caches with torch.cat and
 * gathers them in reorder_incremental_state (:407-420); here the cache is written once per step and a beam
 * reorder moves only the ancestry table, through which the kernel gathers the keys.
 *   q        [tgt_len * bsz, D] with row pitch ldq elements (even), row r = i * bsz + b, already scaled by
 *            head_dim^-0.5 (:209); usually a view of the cache's q columns
 *   cache    [>= n_keys, R, 3D] time-major, one [R, 3D] slab per step: columns [0, D) q, [D, 2D) k,
 *            [2D, 3D) v; R = cache rows per step (the hypothesis count at step 0)
 *   anc      [>= n_keys, bsz] int32 or NULL (identity): anc[s * bsz + b] is the cache row that holds, at step s,
 *            the ancestor of hypothesis b.  An entry outside [0, R) is a masked key.
 *   key_padding [>= n_keys, R] uint8 (1 = padding key, :330-335) indexed by (step, cache row), or NULL
 *   mode     FBKST_SA_INCREMENTAL: tgt_len == 1, the query of row b sees keys 0 .. n_keys-1;
 *            FBKST_SA_FULL: n_keys == tgt_len, every query sees every key;
 *            FBKST_SA_CAUSAL: n_keys == tgt_len, query i sees keys 0 .. i (fairseq's future mask)
 *   out      [tgt_len * bsz, D] (heads concatenated; input of out_proj, :353)
 *   attn_w   w_mode 0: unused; 1: [bsz, tgt_len, n_keys] fp32 averaged over heads (:355-362);
 *            2: [H, bsz, tgt_len, n_keys] fp32 per head.  Masked and future keys get exactly 0.
 * A query whose visible keys are all masked gets a zero output row and zero weights (the reference would
 * produce NaN), as in fbkst_xattn_fwd.  D = 64 * H, H <= 16; 4 * (n_keys * (H + 1) + 64 * H) bytes of shared
 * memory must fit in 200 KB (n_keys <= 2948 at H = 16, <= 5632 at H = 8). */
int fbkst_dec_self_attn_fwd(const void* q, int64_t ldq, const void* cache, const int32_t* anc,
                            const uint8_t* key_padding, void* out, float* attn_w, int w_mode, int mode,
                            int n_keys, int R, int bsz, int tgt_len, int H, fbkst_stream_t stream);
/* fbkst_dec_self_attn_fwd with fp32 q, cache and out: the fp32-accurate decode path.  Same kernel body,
 * fp32 FMA and softmax; every other argument as above. */
int fbkst_dec_self_attn_fwd_f32(const float* q, int64_t ldq, const float* cache, const int32_t* anc,
                                const uint8_t* key_padding, float* out, float* attn_w, int w_mode, int mode,
                                int n_keys, int R, int bsz, int tgt_len, int H, fbkst_stream_t stream);

/* ---- weight preparation (fp32 master parameters -> kernel operand formats) ----------------- */
/* dst[i] = bf16(src[i] * scale) */
int fbkst_cast_bf16(const float* src, void* dst, int64_t n, float scale, fbkst_stream_t stream);
/* conv2 weight [C,C,3,3] fp32 -> [9][C][C] fp16 (tap, out, in) */
int fbkst_prep_conv2_weight(const float* w, void* w_taps, int C, fbkst_stream_t stream);
/* fc3 weight [D, C*F2] (flatten c*F2+f) fp32 -> [D, F2*C] (flatten f*C+c) fp16
 * (the A operand of fc3 is conv2's fp16 output: call fbkst_linear_bf16 with FBKST_EPI_AB_F16) */
int fbkst_prep_fc3_weight(const float* w, void* w_perm, int D, int C, int F2,
                          fbkst_stream_t stream);
/* BatchNorm eval affine: scale = gamma / sqrt(var + eps), shift = beta - mean * scale */
int fbkst_prep_bn_affine(const float* gamma, const float* beta, const float* mean,
                         const float* var, float eps, float* scale, float* shift, int C,
                         fbkst_stream_t stream);

/* =====================================================================================================
 * Training side (scope row T: cfg4).  The reference has no backward code: every gradient below is what
 * torch.autograd derives from the Python calls cited.  Gradients are bf16 GEMM operands with fp32
 * accumulation; parameter gradients are returned in fp32 in the reference's parameter layout.
 * Dropout masks are regenerated from (seed, site, element position), never stored.
 * ===================================================================================================== */

/* x1 = residual + dropout(y, p);  ln_out = LayerNorm(x1) in bf16 (skipped when ln_out == NULL).
 * replaces fairseq/modules/transformer_layer.py:120-122 / :133-135 (F.dropout + residual add) fused with
 * the next sub-layer's LayerNorm (:108-110 / :126-128), and conv_transformer.py:229-232 with residual == NULL.
 * y, residual, x1 [M, D] fp32 (x1 may be NULL); D a multiple of 128. */
int fbkst_dropout_add_ln(const float* y, const float* residual, float* x1, void* ln_out_bf16, const float* gamma,
                         const float* beta, float eps, int M, int D, float p, uint64_t seed, int site,
                         fbkst_stream_t stream);

/* LayerNorm backward (autograd of fairseq/modules/layer_norm.py:29-32): dx (+)= dLN(dy; x, gamma);
 * partial [fbkst_ln_bwd_blocks(M), 2, D] fp32 receives per-block (dgamma | dbeta) sums, to be reduced with
 * fbkst_reduce_sum.  accumulate != 0: dx already holds the residual branch's gradient. */
int fbkst_ln_bwd_blocks(int M);
int fbkst_ln_bwd(const float* dy, const float* x, const float* gamma, float* dx, int accumulate, float* partial,
                 float eps, int M, int D, fbkst_stream_t stream);

/* Gradient preparation for a linear layer's backward: from g [M, N] (g_is_f32: 0 bf16, 1 fp32, 2 IEEE fp16;
 * pitch ldg; optional row
 * remap in_row(m) = (m % remap_inner) * remap_outer + m / remap_inner) produce
 *   v = g, zeroed where the saved activation act[m, n] <= 0 (ReLU backward) and scaled by act_scale,
 *       multiplied by the regenerated dropout keep-scale of element (in_row(m), n) of a [*, dp_cols] tensor;
 *   gb [M, n_pad] bf16 (pitch ldb; columns N..n_pad-1 zero)   -- A operand of the dgrad GEMM        (optional)
 *   gT [N, M] bf16 (pitch ldt)                                 -- A operand of the wgrad GEMM        (optional)
 *   colsum [ceil(M/64), ld_cs] fp32 per-row-tile column sums   -- bias gradient after fbkst_reduce_sum (optional)
 * replaces the autograd of F.relu / F.dropout / F.linear's bias (transformer_layer.py:120-135). */
int fbkst_grad_prep(const void* g, int g_is_f32, int64_t ldg, const void* act_bf16, int64_t lda, float act_scale,
                    int remap_inner, int remap_outer, void* gb, int64_t ldb, int n_pad, void* gT, int64_t ldt,
                    float* colsum, int ld_cs, int M, int N, float p, uint64_t seed, int site, int dp_cols,
                    fbkst_stream_t stream);

/* out[r, c] = scale * sum_{g < G} in[g * g_stride + r * ldi + c]  (fixed summation order) */
int fbkst_reduce_sum(const float* in, int G, int64_t g_stride, int rows, int cols, int64_t ldi, float* out,
                     int64_t ldo, float scale, fbkst_stream_t stream);

/* The same for many independent reductions in ONE launch (a training step has ~120 of them: bias gradients,
 * split-K slices of the weight-gradient GEMMs, LayerNorm parameter gradients -- all consumed only when the
 * backward returns).  `descs` is a HOST array; it is copied into the kernel parameters, so it may be reused
 * as soon as the call returns. */
typedef struct {
  const float* in;
  float* out;
  int64_t g_stride, ldi, ldo;
  int32_t G, rows, cols;
  float scale;
} fbkst_reduce_desc_t;
int fbkst_reduce_sum_batch(const fbkst_reduce_desc_t* descs, int n, fbkst_stream_t stream);

/* Many (bf16 copy, transposed bf16 copy) jobs in ONE launch: job i reads src [rows, cols] (src_type 0 bf16,
 * 1 fp32, 2 IEEE fp16; pitch ld_src elements) and writes copy [rows, cols] bf16 (pitch ld_copy; optional) and
 * transposed [cols, rows] bf16 (pitch ld_transposed; optional).  Used for the per-step operand copies of the
 * fp32 master weights (what autocast / `.half()` does per nn.Linear in the reference's fp16 training) and for
 * the token-contiguous activation copies of the weight-gradient GEMMs.  `descs` is a HOST array (see above);
 * `reserved` is ignored on input. */
typedef struct {
  const void* src;
  void* copy;
  void* transposed;
  int64_t ld_src, ld_copy, ld_transposed;
  int32_t rows, cols, src_type, reserved;
} fbkst_prep_desc_t;
int fbkst_prep_batch(const fbkst_prep_desc_t* descs, int n, fbkst_stream_t stream);

/* Weight gradient of a linear layer: dW[n, k] = sum_m gT[n, m] xT[k, m] (fp32), split-K over the tokens on
 * the CTA-pair tcgen05 kernel + fixed-order reduction.  workspace: fbkst_linear_wgrad_workspace() floats. */
long long fbkst_linear_wgrad_workspace(int n_out, int k_in, int tokens);
int fbkst_linear_wgrad_bf16(const void* gT, int64_t ldg, const void* xT, int64_t ldx, float* workspace, float* dW,
                            int64_t lddw, int n_out, int k_in, int tokens, fbkst_stream_t stream);
/* The same product from the operands' NATURAL layouts (no transposed copies): g [tokens, n_out] bf16 (pitch
 * ldg), x [tokens, k_in] bf16 (pitch ldx; x_is_f16 must be 0: one MMA takes both operands in one format); both
 * 16-byte aligned with pitches % 8 == 0.
 * The tensor cores read both operands MN-major straight from their TMA tiles. */
int fbkst_linear_wgrad_nt(const void* g, int64_t ldg, const void* x, int64_t ldx, int x_is_f16, float* workspace,
                          float* dW, int64_t lddw, int n_out, int k_in, int tokens, fbkst_stream_t stream);
/* Only the split-K GEMM of fbkst_linear_wgrad_bf16: the slices stay in `workspace` as [*splits][ceil32(n_out)][ceil8(k_in)]
 * fp32 and the caller reduces them (fbkst_reduce_sum / fbkst_reduce_sum_batch) when it needs dW. */
int fbkst_linear_wgrad_slices_bf16(const void* gT, int64_t ldg, const void* xT, int64_t ldx, float* workspace,
                                   int n_out, int k_in, int tokens, int* splits, fbkst_stream_t stream);

/* Self-attention for training (local_attention.py:115-139 incl. F.dropout on the probabilities, :136):
 * qkv [L*B, 3*H*64] bf16 UNSCALED (the kernel applies head_dim^-0.5, :98); out [L*B, H*64] bf16;
 * lse [B*H, L] fp32 (log2 domain) is kept for the backward.  Query rows t >= lengths[b] give zeros. */
int fbkst_attention_train_fwd(const void* qkv, void* out, float* lse, const int32_t* lengths, int L, int B, int H,
                              int log_penalty, float dropout_p, uint64_t seed, int site, fbkst_stream_t stream);
/* delta[m, h] = sum_d dO[m, h*64+d] * O[m, h*64+d]  (m = t*B+b) */
int fbkst_attn_delta(const void* dO, const void* O, float* delta, int M, int H, fbkst_stream_t stream);
/* dqkv [L*B, 3*H*64] bf16 = autograd of the call above w.r.t. q, k, v given dO [L*B, H*64] bf16: scores are
 * recomputed tile by tile on tcgen05 (no L x L buffer); rows t >= lengths[b] get zero gradient. */
int fbkst_attention_train_bwd(const void* qkv, const void* dO, const float* lse, const float* delta, void* dqkv,
                              const int32_t* lengths, int L, int B, int H, int log_penalty, float dropout_p,
                              uint64_t seed, int site, fbkst_stream_t stream);

/* CTC-compression backward (conv_transformer.py:290: x.bmm(W) with W constant):
 * dx[t*B+b, :] = weight[t, b] * dout[seg_id[t, b]*B + b, :], zero for padded frames. */
int fbkst_ctc_compress_bwd(const float* dout, const int32_t* seg_id, const float* weight, float* dx, int L, int B,
                           int D, fbkst_stream_t stream);

/* in-place dropout of `numel` (multiple of 4) bf16 / fp32 elements (F.dropout, transformer_layer.py:133) */
int fbkst_dropout_inplace(void* x, int is_f32, int64_t numel, float p, uint64_t seed, int site,
                          fbkst_stream_t stream);

/* ---- next row N1, backward: F.ctc_loss(log_softmax(logits), ..., "sum", zero_infinity=True) differentiated
 * w.r.t. the logits (criterions/CTC_loss.py:143-151 under autograd).  dlogits [L*B, ldd] fp32 =
 * grad_loss[0] * (softmax - occupancies) for frames t < in_lengths[b], zero elsewhere and for utterances
 * with an infeasible alignment.  grad_loss: DEVICE scalar.  alpha_ws: fbkst_ctc_loss_bwd_workspace() floats. */
long long fbkst_ctc_loss_bwd_workspace(int L, int B, int Umax);
int fbkst_ctc_loss_bwd(const void* logits, int logits_dtype, int64_t ldv, const float* lse,
                       const int32_t* in_lengths, const int64_t* targets, int64_t ldt,
                       const int32_t* target_lengths, int blank, const float* grad_loss, float* alpha_ws,
                       float* dlogits, int64_t ldd, int L, int B, int V, int Umax, fbkst_stream_t stream);

/* ---- conv front end, training (conv_transformer.py:203-214).  Activations channels-last [pixels, C], fp16 in
 * the forward, bf16 gradients; pixels = B*T'*F' of the PADDED batch (the reference does not mask: SURVEY F5). */
int fbkst_bn_partial_blocks(void); /* rows of the `partial` scratch buffers below */
/* nn.BatchNorm2d in training mode, statistics half: per-channel batch mean / biased variance of y (the ReLU
 * output), running-stat update (momentum; unbiased variance; running_* may be NULL), mean / rstd for the
 * backward and the affine (scale, shift) for fbkst_bn_apply.  partial: [fbkst_bn_partial_blocks(), 2, C]. */
int fbkst_bn_batch_stats(const void* y_f16, int64_t pixels, int C, const float* gamma, const float* beta, float eps,
                         float momentum, float* running_mean, float* running_var, float* mean, float* rstd,
                         float* scale, float* shift, float* partial, fbkst_stream_t stream);
/* y = dropout(scale[c] * x + shift[c], p)   (BatchNorm affine + F.dropout(p = max(dropout, .1)), :212-214) */
int fbkst_bn_apply(const void* x_f16, void* y_f16, const float* scale, const float* shift, int64_t pixels, int C,
                   float p, uint64_t seed, int site, fbkst_stream_t stream);
/* autograd of dropout(BatchNorm(relu(z))) w.r.t. z: dz [pixels, C] bf16 from dy [pixels, C] bf16 and the saved
 * ReLU output; batch_stats != 0: training-mode BatchNorm (mean / rstd of the batch), else running statistics.
 * sums [2, C] fp32 receives (dbeta | dgamma).  With running statistics (batch_stats == 0) sums and partial may be
 * NULL: the parameter reduction is skipped (frozen BatchNorm). */
int fbkst_bn_relu_bwd(const void* dy_bf16, const void* relu_out_f16, const float* gamma, const float* mean,
                      const float* rstd, int batch_stats, void* dz_bf16, float* sums, float* partial,
                      int64_t pixels, int C, float p, uint64_t seed, int site, fbkst_stream_t stream);
/* conv2 weight-gradient operand: colT [(tap, ci), pixel] bf16 (pitch ldt) from conv1's output y1 [B,T1,F1,C] fp16 */
int fbkst_conv2_im2col_t(const void* y1_f16, void* colT_bf16, int64_t ldt, int B, int T1, int F1, int C,
                         fbkst_stream_t stream);
/* conv2 input gradient: dy1 [B,T1,F1,C] bf16 = gather-sum over taps of dcol [B*T2*F2, 9*C] bf16 (= dz2 @ W2) */
int fbkst_conv2_col2im(const void* dcol_bf16, void* dy1_bf16, int B, int T1, int F1, int C, fbkst_stream_t stream);
/* conv1 weight + bias gradient: dw1b [C, 10] fp32 = (dW1[co, kh*3+kw] | db1[co]) from dz1 [B,T1,F1,C] bf16 and
 * the input batch x [B,T,F] fp32.  partial: [fbkst_bn_partial_blocks(), C, 10]. */
int fbkst_conv1_wgrad(const void* dz1_bf16, const float* x, float* dw1b, float* partial, int B, int T, int F, int C,
                      fbkst_stream_t stream);
/* conv1 input gradient: dx [B,T,F] fp32 = sum over the taps (stride 2, padding 1) of w1 [C, 9] fp32 (= the
 * Conv2d weight [C,1,3,3]) times dz1 [B,T1,F1,C] bf16, T1 = (T+1)/2, F1 = (F+1)/2.  Every input position gets its
 * gradient, padded frames included; fixed summation order (bit-identical across calls). */
int fbkst_conv1_dgrad(const void* dz1_bf16, const float* w1, float* dx, int B, int T, int F, int C,
                      fbkst_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* FBKST_B200_H_ */
