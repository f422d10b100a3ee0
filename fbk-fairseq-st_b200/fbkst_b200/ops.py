"""Tensor-level wrappers over the C ABI.  PyTorch is plumbing here: it owns device memory and the
current stream; all arithmetic happens in ``libfbkst_b200.so``.  Every wrapper raises if the
library or the GPU is missing (no fallback)."""
import torch

from . import _lib
from ._lib import (BF16, CTC_STRATEGY, EPI_AB_F16, EPI_OUT_F32, EPI_POSEMB, EPI_RELU, EPI_ROW_REMAP, F32, SA_CAUSAL,
                   SA_FULL, SA_INCREMENTAL, check)

LAUNCHES = 0  # kernels launched through this module (bench.py reports it as gpu_launches)


def _count(n=1):
    global LAUNCHES
    LAUNCHES += n


try:  # raw handle of the current stream of the current device: two C calls (~0.3 us) instead of the
    # torch.cuda.current_stream() Python path (~5 us; 400+ launches per training step go through here)
    _raw_stream, _cur_device = torch._C._cuda_getCurrentRawStream, torch._C._cuda_getDevice
except AttributeError:  # pragma: no cover
    _raw_stream = _cur_device = None


def _stream():
    if _raw_stream is not None:
        return _raw_stream(_cur_device())
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _req(t, dtype, name):
    if not (isinstance(t, torch.Tensor) and t.is_cuda):
        raise ValueError("fbkst_b200.%s: expected a CUDA tensor" % name)
    if t.dtype != dtype:
        raise ValueError("fbkst_b200.%s: expected %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("fbkst_b200.%s: tensor must be contiguous" % name)
    return t


def cmvn(x, lengths, out=None):
    """apply_mv_norm on a padded batch: x [B,T,F] fp32, lengths [B] int32."""
    lib = _lib.require_device()
    _req(x, torch.float32, "cmvn.x"); _req(lengths, torch.int32, "cmvn.lengths")
    B, T, Fd = x.shape
    out = torch.empty_like(x) if out is None else out
    ws = torch.empty(B * Fd * 2, dtype=torch.float64, device=x.device)
    check(lib.fbkst_cmvn_f32(x.data_ptr(), out.data_ptr(), lengths.data_ptr(), B, T, Fd,
                             ws.data_ptr(), _stream()))
    _count(2)
    return out


def collate_cmvn(packed, starts, lengths, T, normalize=True, out=None):
    """Ragged frames [sum(len), F] fp32 + starts [B] int64 + lengths [B] int32 -> padded [B,T,F]
    (zeros beyond each length), per-utterance CMVN applied in the same pass if ``normalize``."""
    lib = _lib.require_device()
    _req(packed, torch.float32, "collate_cmvn.packed"); _req(starts, torch.int64, "collate_cmvn.starts")
    _req(lengths, torch.int32, "collate_cmvn.lengths")
    B, Fd = lengths.numel(), packed.shape[-1]
    out = torch.empty(B, T, Fd, dtype=torch.float32, device=packed.device) if out is None else out
    ws = torch.empty(B * Fd * 2, dtype=torch.float64, device=packed.device) if normalize else None
    check(lib.fbkst_collate_cmvn_f32(packed.data_ptr(), starts.data_ptr(), lengths.data_ptr(),
                                     out.data_ptr(), B, T, Fd, 1 if normalize else 0, _ptr(ws), _stream()))
    _count(2 if normalize else 1)
    return out


def specaugment_(x, bands, n_freq, n_time):
    """In-place SpecAugment masking: x [B,T,F] fp32, bands [B, n_freq+n_time, 2] int32 (start, width)."""
    lib = _lib.require_device()
    _req(x, torch.float32, "specaugment.x"); _req(bands, torch.int32, "specaugment.bands")
    B, T, Fd = x.shape
    if tuple(bands.shape) != (B, n_freq + n_time, 2):
        raise ValueError("fbkst_b200.specaugment: bands must be [B, n_freq+n_time, 2]")
    check(lib.fbkst_specaugment_f32(x.data_ptr(), bands.data_ptr(), B, T, Fd, n_freq, n_time, _stream()))
    _count()
    return x


def time_stretch(x, windows, T_out):
    """x [B,T,F] fp32, windows [n,4] int32 (first, last, count, flat out offset) -> (out [B,T_out,F],
    ids [B,T_out] int32, -1 beyond the new length)."""
    lib = _lib.require_device()
    _req(x, torch.float32, "time_stretch.x"); _req(windows, torch.int32, "time_stretch.windows")
    B, T, Fd = x.shape
    ids = torch.empty(B, T_out, dtype=torch.int32, device=x.device)
    out = torch.empty(B, T_out, Fd, dtype=torch.float32, device=x.device)
    check(lib.fbkst_time_stretch_f32(x.data_ptr(), windows.data_ptr(), windows.shape[0], ids.data_ptr(),
                                     out.data_ptr(), B, T, T_out, Fd, _stream()))
    _count(2)
    return out, ids


def conv1_relu_bn(x, w, bias, scale, shift):
    lib = _lib.require_device()
    _req(x, torch.float32, "conv1.x")
    B, T, Fd = x.shape
    C = w.shape[0]
    y = torch.empty(B, (T + 1) // 2, (Fd + 1) // 2, C, dtype=torch.float16, device=x.device)
    check(lib.fbkst_conv1_relu_bn(x.data_ptr(), _req(w, torch.float32, "conv1.w").data_ptr(),
                                  bias.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                                  y.data_ptr(), B, T, Fd, C, _stream()))
    _count()
    return y


def conv2_relu_bn(x, w_taps, bias, scale, shift):
    lib = _lib.require_device()
    _req(x, torch.float16, "conv2.x"); _req(w_taps, torch.float16, "conv2.w_taps")
    B, T1, F1, C = x.shape
    y = torch.empty(B, (T1 + 1) // 2, (F1 + 1) // 2, C, dtype=torch.float16, device=x.device)
    check(lib.fbkst_conv2_relu_bn(x.data_ptr(), w_taps.data_ptr(), bias.data_ptr(),
                                  scale.data_ptr(), shift.data_ptr(), y.data_ptr(), B, T1, F1, C,
                                  _stream()))
    _count()
    return y


def conv1_relu_bn_planes(x, w, bias, scale, shift):
    """conv1 -> four (t1, f1)-parity planes [4, B, ceil(T1/2), ceil(F1/2), C] bf16 (see the header)."""
    lib = _lib.require_device()
    _req(x, torch.float32, "conv1.x")
    B, T, Fd = x.shape
    C = w.shape[0]
    T1, F1 = (T + 1) // 2, (Fd + 1) // 2
    y = torch.empty(4, B, (T1 + 1) // 2, (F1 + 1) // 2, C, dtype=torch.float16, device=x.device)
    check(lib.fbkst_conv1_relu_bn_planes(x.data_ptr(), _req(w, torch.float32, "conv1.w").data_ptr(),
                                         bias.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                                         y.data_ptr(), B, T, Fd, C, _stream()))
    _count()
    return y


def conv2_relu_bn_planes(x_planes, T1, F1, w_taps, bias, scale, shift):
    """conv2 over the plane layout of ``conv1_relu_bn_planes``; output as ``conv2_relu_bn``."""
    lib = _lib.require_device()
    _req(x_planes, torch.float16, "conv2.x_planes"); _req(w_taps, torch.float16, "conv2.w_taps")
    four, B, TH, FH, C = x_planes.shape
    if four != 4 or TH != (T1 + 1) // 2 or FH != (F1 + 1) // 2:
        raise ValueError("conv2_relu_bn_planes: plane shape %s does not match T1=%d F1=%d"
                         % (tuple(x_planes.shape), T1, F1))
    y = torch.empty(B, TH, FH, C, dtype=torch.float16, device=x_planes.device)
    check(lib.fbkst_conv2_relu_bn_planes(x_planes.data_ptr(), w_taps.data_ptr(), bias.data_ptr(),
                                         scale.data_ptr(), shift.data_ptr(), y.data_ptr(), B, T1, F1, C,
                                         _stream()))
    _count()
    return y


def linear(a, w, bias=None, relu=False, residual=None, out_dtype=torch.bfloat16, out=None,
           remap=None, posemb=None, rows_limit=None):
    """out = epi(a @ w.T).  a [M,K] bf16, w [N,K] bf16 (or both fp16), bias [N] fp32, residual [M,N] fp32.
    remap=(inner, outer): out row = (m % inner)*outer + m // inner.
    posemb=(table [P,N] fp32, lengths [outer] int32): adds table[pos(m)] (needs remap dims).
    rows_limit=(count [1] int32 device tensor, mult): only rows < count*mult are computed."""
    lib = _lib.require_device()
    if a.dtype == torch.float16:  # the conv front end's operands are IEEE fp16 (conv2 output x fc3 weight)
        _req(a, torch.float16, "linear.a"); _req(w, torch.float16, "linear.w")
    else:
        _req(a, torch.bfloat16, "linear.a"); _req(w, torch.bfloat16, "linear.w")
    M, K = a.shape
    N = w.shape[0]
    if w.shape[1] != K:
        raise ValueError("fbkst_b200.linear: K mismatch %s vs %s" % (tuple(a.shape), tuple(w.shape)))
    flags = (EPI_RELU if relu else 0) | (EPI_OUT_F32 if out_dtype == torch.float32 else 0) | \
        (EPI_AB_F16 if a.dtype == torch.float16 else 0)
    inner = outer = 0
    lengths = None
    res, ldr = residual, 0
    if remap is not None:
        inner, outer = remap
        flags |= EPI_ROW_REMAP
    if posemb is not None:
        res, lengths = posemb
        flags |= EPI_POSEMB
    if res is not None:
        _req(res, torch.float32, "linear.residual")
        ldr = res.stride(0)
    if out is None:
        # rows start on 128-byte lines when N is not already a multiple of 8: the epilogue's 128-byte TMA store
        # boxes then map to whole lines (V = 8005 logits: pitch 8032 instead of 8008)
        ldo = N if N % 8 == 0 else ((N + 31) // 32 * 32 if out_dtype == torch.float32 else (N + 63) // 64 * 64)
        out = torch.empty(M, ldo, dtype=out_dtype, device=a.device)
        if ldo != N:
            out = out[:, :N]
    if out.dtype != out_dtype or out.stride(-1) != 1:
        raise ValueError("fbkst_b200.linear: bad out tensor")
    check(lib.fbkst_linear_bf16(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), _ptr(bias),
                                _ptr(res), ldr, out.data_ptr(), out.stride(0), M, N, K, flags,
                                inner, outer, _ptr(lengths),
                                _ptr(rows_limit[0]) if rows_limit else 0,
                                rows_limit[1] if rows_limit else 0, _stream()))
    _count()
    return out


def linear_ln(a, w, bias=None, relu=False, residual=None, out_dtype=torch.bfloat16, out=None,
              stats_in=None, ln_eps=1e-5, ln_out=None, rows_limit=None):
    """``linear`` with the reference's pre-LayerNorm folded in (fbkst_linear_ln_bf16).
    Consumer side: ``stats_in`` [M, ceil(K/128), 2] fp32 (per-row slice statistics of the LayerNorm
    input whose bf16 copy is ``a``); ``w``/``bias`` are the folded W'' / c of ``fold_layernorm``.
    Producer side (needs ``residual``): ``ln_out=(xb, stats)`` receives bf16(out) and the slice
    statistics of out; pass ``ln_out=True`` to allocate them.  Returns out, or (out, xb, stats)."""
    lib = _lib.require_device()
    _req(a, torch.bfloat16, "linear_ln.a"); _req(w, torch.bfloat16, "linear_ln.w")
    M, K = a.shape
    N = w.shape[0]
    if w.shape[1] != K:
        raise ValueError("fbkst_b200.linear_ln: K mismatch %s vs %s" % (tuple(a.shape), tuple(w.shape)))
    flags = (EPI_RELU if relu else 0) | (EPI_OUT_F32 if out_dtype == torch.float32 else 0)
    ldr = 0
    if residual is not None:
        _req(residual, torch.float32, "linear_ln.residual")
        ldr = residual.stride(0)
    if out is None:
        ldo = (N + 7) // 8 * 8
        out = torch.empty(M, ldo, dtype=out_dtype, device=a.device)
        if ldo != N:
            out = out[:, :N]
    if out.dtype != out_dtype or out.stride(-1) != 1:
        raise ValueError("fbkst_b200.linear_ln: bad out tensor")
    xb = st = None
    if ln_out is not None:
        if ln_out is True:
            ln_out = (torch.empty(M, N, dtype=torch.bfloat16, device=a.device),
                      torch.empty(M, (N + 127) // 128, 2, dtype=torch.float32, device=a.device))
        xb, st = ln_out
        _req(xb, torch.bfloat16, "linear_ln.xb"); _req(st, torch.float32, "linear_ln.stats")
        if xb.shape != (M, N) or st.numel() < M * ((N + 127) // 128) * 2:
            raise ValueError("fbkst_b200.linear_ln: bad ln_out buffers")
    if stats_in is not None:
        _req(stats_in, torch.float32, "linear_ln.stats_in")
        if stats_in.numel() < M * ((K + 127) // 128) * 2:
            raise ValueError("fbkst_b200.linear_ln: stats_in too small")
    check(lib.fbkst_linear_ln_bf16(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), _ptr(bias),
                                   _ptr(residual), ldr, out.data_ptr(), out.stride(0), M, N, K, flags,
                                   _ptr(stats_in), float(ln_eps), _ptr(xb), xb.stride(0) if xb is not None else 0,
                                   _ptr(st), _ptr(rows_limit[0]) if rows_limit else 0,
                                   rows_limit[1] if rows_limit else 0, _stream()))
    _count()
    return out if ln_out is None else (out, xb, st)


def row_stats_cast(x, out=None, rows_limit=None):
    """x [M,D] fp32 -> (bf16(x), slice statistics [M, D/128, 2]) for the folded LayerNorm."""
    lib = _lib.require_device()
    _req(x, torch.float32, "row_stats_cast.x")
    M, D = x.shape
    if out is None:
        out = (torch.empty(M, D, dtype=torch.bfloat16, device=x.device),
               torch.empty(M, (D + 127) // 128, 2, dtype=torch.float32, device=x.device))
    xb, st = out
    check(lib.fbkst_row_stats_cast(x.data_ptr(), xb.data_ptr(), st.data_ptr(), M, D,
                                   _ptr(rows_limit[0]) if rows_limit else 0,
                                   rows_limit[1] if rows_limit else 0, _stream()))
    _count()
    return xb, st


def embed_remap_stats(src, L, B, table=None, lengths=None):
    """fc3 output [B*L, D] fp32 in (b, t) row order -> time-major x [L*B, D] fp32 (+ sinusoidal positions
    from ``table`` masked by ``lengths``: conv_transformer.py:225-229), bf16(x) and the slice statistics
    of ``row_stats_cast`` in one pass."""
    lib = _lib.require_device()
    _req(src, torch.float32, "embed_remap_stats.src")
    M, D = src.shape
    if M != L * B:
        raise ValueError("embed_remap_stats: src has %d rows, expected L*B = %d" % (M, L * B))
    if table is not None:
        _req(table, torch.float32, "embed_remap_stats.table")
        _req(lengths, torch.int32, "embed_remap_stats.lengths")
        if table.shape[0] < L + 1 or table.shape[1] != D:
            raise ValueError("embed_remap_stats: position table too small")
    x = torch.empty(M, D, dtype=torch.float32, device=src.device)
    xb = torch.empty(M, D, dtype=torch.bfloat16, device=src.device)
    st = torch.empty(M, (D + 127) // 128, 2, dtype=torch.float32, device=src.device)
    check(lib.fbkst_embed_remap_stats(src.data_ptr(), _ptr(table), table.stride(0) if table is not None else 0,
                                      _ptr(lengths) if table is not None else 0, x.data_ptr(), xb.data_ptr(),
                                      st.data_ptr(), L, B, D, _stream()))
    _count()
    return x, xb, st


def fold_layernorm(w, b, gamma, beta, row_scale=None):
    """Weights of ``linear_ln``'s consumer side: W''[n,k] = gamma[k] W[n,k] - mean_k(gamma[k] W[n,k])
    (bf16) and c[n] = b[n] + sum_k beta[k] W[n,k] (fp32), so that LN(x) W^T + b == rstd(x) * (x W''^T)
    + c.  ``row_scale`` [N] optionally scales output rows (the q rows of the in-projection).
    One-time parameter preparation (fp64 on the device), like ``prep_*``."""
    w64, g64 = w.detach().double(), gamma.detach().double()
    wg = w64 * g64[None, :]
    wg = wg - wg.mean(dim=1, keepdim=True)
    c = b.detach().double() + w64 @ beta.detach().double()
    if row_scale is not None:
        wg = wg * row_scale.double()[:, None]
        c = c * row_scale.double()
    return cast_bf16(wg.float().contiguous()), c.float().contiguous()


def layernorm(x, gamma, beta, out_dtype=torch.bfloat16, eps=1e-5, out=None, rows_limit=None):
    lib = _lib.require_device()
    _req(x, torch.float32, "layernorm.x")
    M, D = x.shape
    y = torch.empty(M, D, dtype=out_dtype, device=x.device) if out is None else out
    check(lib.fbkst_layernorm(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(),
                              F32 if out_dtype == torch.float32 else BF16, M, D, eps,
                              _ptr(rows_limit[0]) if rows_limit else 0,
                              rows_limit[1] if rows_limit else 0, _stream()))
    _count()
    return y


def attention(qkv, lengths, L, B, H, log_penalty=True, out=None, q_limit=None):
    """qkv [L*B, 3*H*64] bf16 (row t*B+b) -> [L*B, H*64] bf16.  ``q_limit`` (device int32 [1]): the caller
    only reads query rows t < q_limit; fully padded query tiles beyond it are not even zero-filled."""
    lib = _lib.require_device()
    _req(qkv, torch.bfloat16, "attention.qkv"); _req(lengths, torch.int32, "attention.lengths")
    if qkv.shape != (L * B, 3 * H * 64):
        raise ValueError("fbkst_b200.attention: qkv shape %s != (%d, %d)" %
                         (tuple(qkv.shape), L * B, 3 * H * 64))
    if out is None:
        out = torch.empty(L * B, H * 64, dtype=torch.bfloat16, device=qkv.device)
    if q_limit is not None:
        _req(q_limit, torch.int32, "attention.q_limit")
        check(lib.fbkst_attention_fwd_limited(qkv.data_ptr(), out.data_ptr(), lengths.data_ptr(), L, B, H,
                                              1 if log_penalty else 0, q_limit.data_ptr(), _stream()))
    else:
        check(lib.fbkst_attention_fwd(qkv.data_ptr(), out.data_ptr(), lengths.data_ptr(), L, B, H,
                                      1 if log_penalty else 0, _stream()))
    _count()
    return out


def sinusoidal_table(rows, D, device):
    lib = _lib.require_device()
    t = torch.empty(rows, D, dtype=torch.float32, device=device)
    check(lib.fbkst_sinusoidal_table(t.data_ptr(), rows, D, _stream()))
    _count()
    return t


def lengths_to_mask(lengths, L):
    """-> (mask [B,L] bool, any_pad [1] int32 device tensor)."""
    lib = _lib.require_device()
    _req(lengths, torch.int32, "lengths_to_mask.lengths")
    B = lengths.numel()
    mask = torch.empty(B, L, dtype=torch.uint8, device=lengths.device)
    any_pad = torch.empty(1, dtype=torch.int32, device=lengths.device)
    check(lib.fbkst_lengths_to_mask(lengths.data_ptr(), mask.data_ptr(), any_pad.data_ptr(), B, L,
                                    _stream()))
    _count()
    return mask.view(torch.bool), any_pad


def subsample_lengths(lengths, times=2):
    """Device-resident lengths [B] int64/int32 -> int32 lengths after ``times`` stride-2 convolutions
    (ceil(n/2) each, conv_transformer.py:213)."""
    lib = _lib.require_device()
    if not lengths.is_cuda or lengths.dtype not in (torch.int64, torch.int32) or not lengths.is_contiguous():
        raise ValueError("fbkst_b200.subsample_lengths: expected a contiguous CUDA int64/int32 vector")
    out = torch.empty(lengths.numel(), dtype=torch.int32, device=lengths.device)
    check(lib.fbkst_subsample_lengths(lengths.data_ptr(), 1 if lengths.dtype == torch.int64 else 0,
                                      out.data_ptr(), lengths.numel(), int(times), _stream()))
    _count()
    return out


def linear_argmax(a, w, bias, lengths, L, B, want_prob=True, want_lse=False, bump=None):
    """ctc_fc with the frame arg-max folded into the GEMM epilogue.  a [L*B, K] bf16, w [V, K] bf16, bias [V]
    fp32.  bump=(labels [L*B] int32, margin): logits[row, labels[row]] += margin before store and arg-max.
    -> (logits [L*B, V] fp32 view of a 128-byte-pitched buffer, labels [L*B] int32, top_prob or None, lse or None)."""
    lib = _lib.require_device()
    _req(a, torch.bfloat16, "linear_argmax.a"); _req(w, torch.bfloat16, "linear_argmax.w")
    _req(lengths, torch.int32, "linear_argmax.lengths")
    M, K = a.shape
    V = w.shape[0]
    if M != L * B or w.shape[1] != K:
        raise ValueError("fbkst_b200.linear_argmax: shape mismatch")
    dev = a.device
    ldo = (V + 31) // 32 * 32
    out = torch.empty(M, ldo, dtype=torch.float32, device=dev)
    chunks = (V + 127) // 128
    partial = torch.empty(M, chunks, 4, dtype=torch.float32, device=dev)
    bl, bm = (None, 0.0) if bump is None else bump
    if bl is not None:
        _req(bl, torch.int32, "linear_argmax.bump labels")
        if bl.numel() != M:
            raise ValueError("fbkst_b200.linear_argmax: bump labels must have L*B entries")
    want_sum = want_prob or want_lse
    check(lib.fbkst_linear_argmax_f32(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), _ptr(bias),
                                      out.data_ptr(), ldo, M, V, K, _ptr(bl), float(bm), 1 if want_sum else 0,
                                      partial.data_ptr(), 0, 0, _stream()))
    labels = torch.empty(M, dtype=torch.int32, device=dev)
    prob = torch.empty(M, dtype=torch.float32, device=dev) if want_prob else None
    lse = torch.empty(M, dtype=torch.float32, device=dev) if want_lse else None
    check(lib.fbkst_ctc_argmax_merge(partial.data_ptr(), chunks, out.data_ptr(), ldo, V, lengths.data_ptr(),
                                     labels.data_ptr(), _ptr(prob), _ptr(lse), L, B, _stream()))
    _count(2)
    return out[:, :V], labels, prob, lse


def ctc_argmax(logits, lengths, L, B, V, want_prob=True):
    """logits [L*B, >=V] bf16/fp32 (possibly a column-narrowed view) -> labels, top_prob."""
    lib = _lib.require_device()
    if logits.dtype not in (torch.bfloat16, torch.float32) or logits.stride(-1) != 1:
        raise ValueError("fbkst_b200.ctc_argmax: logits must be bf16/fp32 with unit column stride")
    labels = torch.empty(L * B, dtype=torch.int32, device=logits.device)
    prob = torch.empty(L * B, dtype=torch.float32, device=logits.device) if want_prob else None
    check(lib.fbkst_ctc_argmax(logits.data_ptr(), BF16 if logits.dtype == torch.bfloat16 else F32,
                               logits.stride(0), lengths.data_ptr(), labels.data_ptr(), _ptr(prob),
                               L, B, V, _stream()))
    _count()
    return labels, prob


def ctc_argmax_lse(logits, lengths, L, B, V, want_prob=False):
    """As ctc_argmax, plus lse[L*B] fp32 = logsumexp of every valid row (0 for padding)."""
    lib = _lib.require_device()
    if logits.dtype not in (torch.bfloat16, torch.float32) or logits.stride(-1) != 1:
        raise ValueError("fbkst_b200.ctc_argmax_lse: logits must be bf16/fp32 with unit column stride")
    labels = torch.empty(L * B, dtype=torch.int32, device=logits.device)
    lse = torch.empty(L * B, dtype=torch.float32, device=logits.device)
    prob = torch.empty(L * B, dtype=torch.float32, device=logits.device) if want_prob else None
    check(lib.fbkst_ctc_argmax_lse(logits.data_ptr(), BF16 if logits.dtype == torch.bfloat16 else F32,
                                   logits.stride(0), lengths.data_ptr(), labels.data_ptr(), _ptr(prob),
                                   lse.data_ptr(), L, B, V, _stream()))
    _count()
    return labels, lse, prob


def ctc_uer(labels, in_lengths, targets, target_lengths, blank, L, B):
    """compute_ctc_uer on device.  labels [L*B] int32 (from ctc_argmax), in_lengths / target_lengths
    [B] int32, targets [B, U] int64 (padded).  -> errors [B] int32, pred_lengths [B] int32,
    totals [2] int64 = (batch_errors, batch_total); nothing is synchronised."""
    lib = _lib.require_device()
    _req(labels, torch.int32, "ctc_uer.labels"); _req(in_lengths, torch.int32, "ctc_uer.in_lengths")
    _req(target_lengths, torch.int32, "ctc_uer.target_lengths")
    if targets.dtype != torch.int64 or targets.dim() != 2 or (targets.numel() and targets.stride(1) != 1):
        raise ValueError("fbkst_b200.ctc_uer: targets must be [B, U] int64 with unit column stride")
    U = targets.shape[1]
    dev = labels.device
    errors = torch.empty(B, dtype=torch.int32, device=dev)
    plen = torch.empty(B, dtype=torch.int32, device=dev)
    totals = torch.empty(2, dtype=torch.int64, device=dev)
    check(lib.fbkst_ctc_uer(labels.data_ptr(), in_lengths.data_ptr(), targets.data_ptr() if U else 0,
                            targets.stride(0) if U else 0, target_lengths.data_ptr(), int(blank),
                            errors.data_ptr(), plen.data_ptr(), totals.data_ptr(), L, B, U, _stream()))
    _count(2)
    return errors, plen, totals


def ctc_loss_fwd(logits, lse, in_lengths, targets, target_lengths, blank, L, B, V):
    """F.ctc_loss(log_softmax(logits), ..., reduction="sum", zero_infinity=True) forward.
    logits [L*B, >=V] bf16/fp32 rows t*B+b, lse from ctc_argmax_lse.  -> nll [B] fp32, loss [1] fp32."""
    lib = _lib.require_device()
    if logits.dtype not in (torch.bfloat16, torch.float32) or logits.stride(-1) != 1:
        raise ValueError("fbkst_b200.ctc_loss_fwd: logits must be bf16/fp32 with unit column stride")
    _req(lse, torch.float32, "ctc_loss_fwd.lse"); _req(in_lengths, torch.int32, "ctc_loss_fwd.in_lengths")
    _req(target_lengths, torch.int32, "ctc_loss_fwd.target_lengths")
    if targets.dtype != torch.int64 or targets.dim() != 2 or (targets.numel() and targets.stride(1) != 1):
        raise ValueError("fbkst_b200.ctc_loss_fwd: targets must be [B, U] int64 with unit column stride")
    U = targets.shape[1]
    nll = torch.empty(B, dtype=torch.float32, device=logits.device)
    loss = torch.empty(1, dtype=torch.float32, device=logits.device)
    check(lib.fbkst_ctc_loss_fwd(logits.data_ptr(), BF16 if logits.dtype == torch.bfloat16 else F32,
                                 logits.stride(0), lse.data_ptr(), in_lengths.data_ptr(),
                                 targets.data_ptr() if U else 0, targets.stride(0) if U else 0,
                                 target_lengths.data_ptr(), int(blank), nll.data_ptr(), loss.data_ptr(),
                                 L, B, V, U, _stream()))
    _count(2)
    return nll, loss


def ctc_segment(labels, top_prob, lengths, strategy, L, B):
    lib = _lib.require_device()
    dev = labels.device
    seg_id = torch.empty(L * B, dtype=torch.int32, device=dev)
    seg_start = torch.empty(L * B, dtype=torch.int32, device=dev)
    weight = torch.empty(L * B, dtype=torch.float32, device=dev)
    new_len = torch.empty(B, dtype=torch.int32, device=dev)
    max_new = torch.empty(1, dtype=torch.int32, device=dev)
    check(lib.fbkst_ctc_segment(labels.data_ptr(), _ptr(top_prob), lengths.data_ptr(),
                                CTC_STRATEGY[strategy], seg_id.data_ptr(), seg_start.data_ptr(),
                                weight.data_ptr(), new_len.data_ptr(), max_new.data_ptr(), L, B,
                                _stream()))
    _count()
    return seg_id, seg_start, weight, new_len, max_new


def ctc_compress(x, seg_id, seg_start, weight, lengths, new_len, max_new, L, B, out=None):
    lib = _lib.require_device()
    _req(x, torch.float32, "ctc_compress.x")
    D = x.shape[-1]
    if out is None:
        out = torch.empty(L * B, D, dtype=torch.float32, device=x.device)
    check(lib.fbkst_ctc_compress(x.data_ptr(), seg_id.data_ptr(), seg_start.data_ptr(), weight.data_ptr(),
                                 lengths.data_ptr(), new_len.data_ptr(), max_new.data_ptr(),
                                 out.data_ptr(), L, B, D, _stream()))
    _count()
    return out


def xattn(q, kv, mask, row_map, S, U, bsz, tgt_len, H, weights=0):
    """Encoder-decoder attention for ``tgt_len * bsz`` query rows over per-utterance K/V.
    q [tgt_len*bsz, D] bf16 (pre-scaled), kv [S, U, 2D] bf16, mask [U, S] bool/uint8 or None,
    row_map [bsz] int32.  weights: 0 none, 1 head-averaged [bsz, tgt_len, S], 2 per head
    [H, bsz, tgt_len, S].  Returns (out [tgt_len*bsz, D] bf16, weights or None)."""
    return _xattn("xattn", torch.bfloat16, q, kv, mask, row_map, S, U, bsz, tgt_len, H, weights)


def xattn_f32(q, kv, mask, row_map, S, U, bsz, tgt_len, H, weights=0):
    """``xattn`` with fp32 q [tgt_len*bsz, D], kv [S, U, 2D] and out (fp32 FMA throughout)."""
    return _xattn("xattn_f32", torch.float32, q, kv, mask, row_map, S, U, bsz, tgt_len, H, weights)


def _xattn(name, dtype, q, kv, mask, row_map, S, U, bsz, tgt_len, H, weights):
    lib = _lib.require_device()
    _req(q, dtype, name + ".q"); _req(kv, dtype, name + ".kv")
    _req(row_map, torch.int32, name + ".row_map")
    D = 64 * H
    if tuple(q.shape) != (tgt_len * bsz, D) or tuple(kv.shape) != (S, U, 2 * D) or row_map.numel() != bsz:
        raise ValueError("fbkst_b200.%s: shape mismatch q %s kv %s row_map %s" %
                         (name, tuple(q.shape), tuple(kv.shape), tuple(row_map.shape)))
    if mask is not None:
        if mask.dtype == torch.bool:
            mask = mask.view(torch.uint8)
        _req(mask, torch.uint8, name + ".mask")
        if tuple(mask.shape) != (U, S):
            raise ValueError("fbkst_b200.%s: mask must be [U, S]" % name)
    out = torch.empty(tgt_len * bsz, D, dtype=dtype, device=q.device)
    w = ws = None
    if weights == 1:
        w = torch.empty(bsz, tgt_len, S, dtype=torch.float32, device=q.device)
        ws = torch.empty(H, bsz, tgt_len, S, dtype=torch.float32, device=q.device)
    elif weights == 2:
        w = torch.empty(H, bsz, tgt_len, S, dtype=torch.float32, device=q.device)
    fn = lib.fbkst_xattn_fwd_f32 if dtype == torch.float32 else lib.fbkst_xattn_fwd
    check(fn(q.data_ptr(), kv.data_ptr(), _ptr(mask), row_map.data_ptr(), out.data_ptr(),
             _ptr(w), _ptr(ws), weights, S, U, bsz, tgt_len, H, _stream()))
    _count(2 if weights == 1 else 1)
    return out, w


def dec_self_attn(q, cache, anc, pad, n_keys, bsz, tgt_len, H, mode=SA_INCREMENTAL, weights=0):
    """Decoder self-attention of ``tgt_len * bsz`` query rows over an append-only cache.
    q [tgt_len*bsz, D] bf16 (pre-scaled; unit column stride, any even row pitch: usually a view of the cache's
    q columns), cache [T_cap, R, 3D] bf16 (per step: q | k | v of R cache rows), anc [>= n_keys, bsz] int32 or
    None (hypothesis b reads cache row anc[s, b] at step s), pad [T_cap, R] bool/uint8 or None (padding keys by
    step and cache row).  mode: SA_INCREMENTAL (tgt_len 1, keys 0..n_keys-1), SA_FULL or SA_CAUSAL (n_keys ==
    tgt_len).  weights: 0 none, 1 head-averaged [bsz, tgt_len, n_keys], 2 per head [H, bsz, tgt_len, n_keys].
    Returns (out [tgt_len*bsz, D] bf16, weights or None)."""
    return _dec_self_attn("dec_self_attn", torch.bfloat16, q, cache, anc, pad, n_keys, bsz, tgt_len, H, mode,
                          weights)


def dec_self_attn_f32(q, cache, anc, pad, n_keys, bsz, tgt_len, H, mode=SA_INCREMENTAL, weights=0):
    """``dec_self_attn`` with fp32 q, cache and out (fp32 FMA throughout)."""
    return _dec_self_attn("dec_self_attn_f32", torch.float32, q, cache, anc, pad, n_keys, bsz, tgt_len, H, mode,
                          weights)


def _dec_self_attn(name, dtype, q, cache, anc, pad, n_keys, bsz, tgt_len, H, mode, weights):
    lib = _lib.require_device()
    _req(cache, dtype, name + ".cache")
    D = 64 * H
    if not (isinstance(q, torch.Tensor) and q.is_cuda and q.dtype == dtype):
        raise ValueError("fbkst_b200.%s.q: expected a CUDA %s tensor" % (name, dtype))
    if q.dim() != 2 or tuple(q.shape) != (tgt_len * bsz, D) or q.stride(1) != 1:
        raise ValueError("fbkst_b200.%s: q must be [tgt_len*bsz, D] = (%d, %d) with unit column stride, got %s" %
                         (name, tgt_len * bsz, D, tuple(q.shape)))
    if cache.dim() != 3 or cache.shape[2] != 3 * D or cache.shape[0] < n_keys:
        raise ValueError("fbkst_b200.%s: cache %s must be [>= %d steps, R, 3D = %d]" %
                         (name, tuple(cache.shape), n_keys, 3 * D))
    R = cache.shape[1]
    if anc is not None:
        _req(anc, torch.int32, name + ".anc")
        if anc.dim() != 2 or anc.shape[0] < n_keys or anc.shape[1] != bsz:
            raise ValueError("fbkst_b200.%s: anc %s must be [>= %d, bsz = %d]" % (name, tuple(anc.shape), n_keys, bsz))
    if pad is not None:
        if pad.dtype == torch.bool:
            pad = pad.view(torch.uint8)
        _req(pad, torch.uint8, name + ".pad")
        if tuple(pad.shape) != tuple(cache.shape[:2]):
            raise ValueError("fbkst_b200.%s: pad must be [T_cap, R] = %s" % (name, tuple(cache.shape[:2])))
    if mode not in (SA_INCREMENTAL, SA_FULL, SA_CAUSAL) or weights not in (0, 1, 2):
        raise ValueError("fbkst_b200.%s: mode %r / weights %r out of range" % (name, mode, weights))
    out = torch.empty(tgt_len * bsz, D, dtype=dtype, device=q.device)
    w = None
    if weights == 1:
        w = torch.empty(bsz, tgt_len, n_keys, dtype=torch.float32, device=q.device)
    elif weights == 2:
        w = torch.empty(H, bsz, tgt_len, n_keys, dtype=torch.float32, device=q.device)
    fn = lib.fbkst_dec_self_attn_fwd_f32 if dtype == torch.float32 else lib.fbkst_dec_self_attn_fwd
    check(fn(q.data_ptr(), q.stride(0), cache.data_ptr(), _ptr(anc), _ptr(pad), out.data_ptr(), _ptr(w), weights,
             mode, n_keys, R, bsz, tgt_len, H, _stream()))
    _count()
    return out, w


def cast_bf16(src, scale=1.0):
    lib = _lib.require_device()
    src = _req(src.contiguous(), torch.float32, "cast_bf16.src")
    dst = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    check(lib.fbkst_cast_bf16(src.data_ptr(), dst.data_ptr(), src.numel(), float(scale), _stream()))
    _count()
    return dst


def prep_conv2_weight(w):
    lib = _lib.require_device()
    w = _req(w.contiguous(), torch.float32, "prep_conv2_weight.w")
    C = w.shape[0]
    out = torch.empty(9, C, C, dtype=torch.float16, device=w.device)
    check(lib.fbkst_prep_conv2_weight(w.data_ptr(), out.data_ptr(), C, _stream()))
    _count()
    return out


def prep_fc3_weight(w, C, F2):
    lib = _lib.require_device()
    w = _req(w.contiguous(), torch.float32, "prep_fc3_weight.w")
    D = w.shape[0]
    out = torch.empty(D, F2 * C, dtype=torch.float16, device=w.device)
    check(lib.fbkst_prep_fc3_weight(w.data_ptr(), out.data_ptr(), D, C, F2, _stream()))
    _count()
    return out


def prep_bn_affine(gamma, beta, mean, var, eps=1e-5):
    lib = _lib.require_device()
    C = gamma.numel()
    scale = torch.empty(C, dtype=torch.float32, device=gamma.device)
    shift = torch.empty(C, dtype=torch.float32, device=gamma.device)
    check(lib.fbkst_prep_bn_affine(gamma.data_ptr(), beta.data_ptr(), mean.data_ptr(),
                                   var.data_ptr(), eps, scale.data_ptr(), shift.data_ptr(), C,
                                   _stream()))
    _count()
    return scale, shift


# ----------------------------------------------------------------- fp32-accurate path (split TF32, DESIGN F)
def linear_f32(a, w, bias=None, relu=False, residual=None, affine=None, out=None, rows_limit=None):
    """out = epi(a @ w.T) on the split-TF32 tensor-core GEMM.  a [M,K] fp32 (unit column stride, pitch % 4 == 0),
    w [N,K] fp32, bias [N] fp32, affine=(scale [N], shift [N]) applied after the ReLU, residual [M,N] fp32.
    rows_limit=(count [1] int32 device tensor, mult): only rows < count*mult are computed."""
    lib = _lib.require_device()
    for t, name in ((a, "a"), (w, "w")):
        if not (t.is_cuda and t.dtype == torch.float32 and t.dim() == 2 and t.stride(1) == 1):
            raise ValueError("fbkst_b200.linear_f32: %s must be a 2-D CUDA fp32 tensor with unit column stride" % name)
    M, K = a.shape
    N = w.shape[0]
    if w.shape[1] != K:
        raise ValueError("fbkst_b200.linear_f32: K mismatch %s vs %s" % (tuple(a.shape), tuple(w.shape)))
    if bias is not None:
        _req(bias, torch.float32, "linear_f32.bias")
    sc, sh = (None, None) if affine is None else affine
    ldr = 0
    if residual is not None:
        if residual.dtype != torch.float32 or residual.stride(1) != 1 or tuple(residual.shape) != (M, N):
            raise ValueError("fbkst_b200.linear_f32: residual must be [M, N] fp32 with unit column stride")
        ldr = residual.stride(0)
    if out is None:
        ldo = (N + 3) // 4 * 4
        out = torch.empty(M, ldo, dtype=torch.float32, device=a.device)
        if ldo != N:
            out = out[:, :N]
    if out.dtype != torch.float32 or out.stride(-1) != 1 or tuple(out.shape) != (M, N):
        raise ValueError("fbkst_b200.linear_f32: bad out tensor")
    check(lib.fbkst_linear_tf32x3(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), _ptr(bias), _ptr(sc),
                                  _ptr(sh), _ptr(residual), ldr, out.data_ptr(), out.stride(0), M, N, K,
                                  1 if relu else 0, _ptr(rows_limit[0]) if rows_limit else 0,
                                  rows_limit[1] if rows_limit else 0, _stream()))
    _count()
    return out


def attention_f32(qkv, lengths, L, B, H, log_penalty=True, out=None, q_limit=None):
    """qkv [L*B, 3*H*64] fp32 (row t*B+b, q pre-scaled) -> [L*B, H*64] fp32 on split-TF32 tensor cores.
    ``q_limit`` as in ``attention``."""
    lib = _lib.require_device()
    _req(qkv, torch.float32, "attention_f32.qkv"); _req(lengths, torch.int32, "attention_f32.lengths")
    if qkv.shape != (L * B, 3 * H * 64):
        raise ValueError("fbkst_b200.attention_f32: qkv shape %s != (%d, %d)" %
                         (tuple(qkv.shape), L * B, 3 * H * 64))
    if out is None:
        out = torch.empty(L * B, H * 64, dtype=torch.float32, device=qkv.device)
    _req(out, torch.float32, "attention_f32.out")
    if q_limit is not None:
        _req(q_limit, torch.int32, "attention_f32.q_limit")
    check(lib.fbkst_attention_tf32x3(qkv.data_ptr(), out.data_ptr(), lengths.data_ptr(), L, B, H,
                                     1 if log_penalty else 0, _ptr(q_limit), _stream()))
    _count()
    return out


def conv1_relu_bn_f32(x, w, bias, scale, shift):
    """x [B,T,F] fp32, w [C,9] fp32 -> y [B,T1,F1,C] fp32 = BN(ReLU(conv1(x)))."""
    lib = _lib.require_device()
    _req(x, torch.float32, "conv1_f32.x"); _req(w, torch.float32, "conv1_f32.w")
    B, T, Fd = x.shape
    C = w.shape[0]
    y = torch.empty(B, (T + 1) // 2, (Fd + 1) // 2, C, dtype=torch.float32, device=x.device)
    check(lib.fbkst_conv1_relu_bn_f32(x.data_ptr(), w.data_ptr(), bias.data_ptr(), scale.data_ptr(),
                                      shift.data_ptr(), y.data_ptr(), B, T, Fd, C, _stream()))
    _count()
    return y


def conv2_relu_bn_f32(y1, w2, bias, scale, shift):
    """y1 [B,T1,F1,C] fp32 -> [B,T2,F2,C] fp32 = BN(ReLU(conv2(y1))): fp32 patches (im2col), then the split-TF32
    GEMM with ``w2`` [C, 9*C] from ``prep_conv2_weight_f32``."""
    lib = _lib.require_device()
    _req(y1, torch.float32, "conv2_f32.y1")
    B, T1, F1, C = y1.shape
    T2, F2 = (T1 + 1) // 2, (F1 + 1) // 2
    col = torch.empty(B * T2 * F2, 9 * C, dtype=torch.float32, device=y1.device)
    check(lib.fbkst_conv2_im2col_f32(y1.data_ptr(), col.data_ptr(), B, T1, F1, C, _stream()))
    _count()
    y = linear_f32(col, w2, bias, relu=True, affine=(scale, shift))
    return y.view(B, T2, F2, C)


def prep_conv2_weight_f32(w):
    """conv2 weight [C,C,3,3] -> [C, 9*C] fp32, column (kt*3 + kf)*C + c (the patch order of conv2_relu_bn_f32)."""
    C = w.shape[0]
    return w.detach().float().permute(0, 2, 3, 1).reshape(C, 9 * C).contiguous()


def prep_fc3_weight_f32(w, C, F2):
    """fc3 weight [D, C*F2] (reference flatten c*F2+f) -> [D, F2*C] fp32 (channels-last flatten f*C+c)."""
    D = w.shape[0]
    return w.detach().float().view(D, C, F2).permute(0, 2, 1).reshape(D, F2 * C).contiguous()


# ------------------------------------------------------------------------------------- training side
# Batched launches: the job tables of fbkst_reduce_sum_batch / fbkst_prep_batch are packed HOST arrays of the
# structs declared in include/fbkst_b200.h (fbkst_reduce_desc_t: 56 bytes, fbkst_prep_desc_t: 64 bytes).
import ctypes as _ct  # noqa: E402
import struct as _struct  # noqa: E402

_REDUCE_FMT, _PREP_FMT = "<QQqqqiiif", "<QQQqqqiiii"
assert _struct.calcsize(_REDUCE_FMT) == 56 and _struct.calcsize(_PREP_FMT) == 64
_SRC_TYPE = {torch.bfloat16: 0, torch.float32: 1, torch.float16: 2}


class _ReduceQueue:
    """Fixed-order reductions whose results are only needed later (bias / weight / LayerNorm parameter
    gradients): collected while ``deferred_reductions()`` is active, launched together by ``flush``."""

    def __init__(self):
        self.buf, self.keep, self.n = bytearray(), [], 0

    def add(self, src, G, g_stride, rows, cols, ldi, out, ldo, scale):
        self.buf += _struct.pack(_REDUCE_FMT, src.data_ptr(), out.data_ptr(), g_stride, ldi, ldo, G, rows, cols, scale)
        self.keep.append((src, out))  # the partial sums must outlive the launch
        self.n += 1

    def flush(self):
        if self.n:
            lib = _lib.require_device()
            raw = (_ct.c_char * len(self.buf)).from_buffer(self.buf)
            check(lib.fbkst_reduce_sum_batch(_ct.addressof(raw), self.n, _stream()))
            _count((self.n + 55) // 56)
            del raw
        self.buf, self.keep, self.n = bytearray(), [], 0


_DEFER = None


class deferred_reductions:
    """``with ops.deferred_reductions():`` -- ``reduce_sum`` calls made inside (directly or by grad_prep / ln_bwd /
    linear_wgrad) are queued and run as one batched launch on exit.  Their outputs must not be read inside."""

    def __enter__(self):
        global _DEFER
        self.prev, _DEFER = _DEFER, _ReduceQueue()
        return _DEFER

    def __exit__(self, *exc):
        global _DEFER
        q, _DEFER = _DEFER, self.prev
        if exc[0] is None:
            q.flush()
        return False


def reduce_sum(src, G, g_stride, rows, cols, ldi, out, ldo, scale=1.0):
    """out[r, c] = scale * sum_g src[g * g_stride + r * ldi + c] (fixed order); queued when deferral is active."""
    if _DEFER is not None:
        _DEFER.add(src, G, g_stride, rows, cols, ldi, out, ldo, scale)
        return
    lib = _lib.require_device()
    check(lib.fbkst_reduce_sum(src.data_ptr(), G, g_stride, rows, cols, ldi, out.data_ptr(), ldo, scale, _stream()))
    _count()


def prep_batch(jobs):
    """jobs: iterable of (src [rows, cols] bf16/fp32/fp16 with unit column stride, copy or None, transposed or
    None); copy [rows, cols] bf16 / transposed [cols, rows] bf16 are 2-D tensors or views with unit column stride
    (pitches taken from their strides).  One launch per 48 jobs."""
    lib = _lib.require_device()
    buf, n = bytearray(), 0
    for src, copy, tr in jobs:
        if src.dim() != 2 or src.stride(1) != 1 or src.dtype not in _SRC_TYPE or not src.is_cuda:
            raise ValueError("fbkst_b200.prep_batch: src must be a 2-D CUDA bf16/fp32/fp16 tensor, unit column stride")
        rows, cols = src.shape
        for t, shp, name in ((copy, (rows, cols), "copy"), (tr, (cols, rows), "transposed")):
            if t is not None and (t.dtype != torch.bfloat16 or tuple(t.shape) != shp or t.stride(1) != 1):
                raise ValueError("fbkst_b200.prep_batch: bad %s tensor" % name)
        buf += _struct.pack(_PREP_FMT, src.data_ptr(), _ptr(copy), _ptr(tr), src.stride(0),
                            copy.stride(0) if copy is not None else 0, tr.stride(0) if tr is not None else 0,
                            rows, cols, _SRC_TYPE[src.dtype], 0)
        n += 1
    if n:
        raw = (_ct.c_char * len(buf)).from_buffer(buf)
        check(lib.fbkst_prep_batch(_ct.addressof(raw), n, _stream()))
        _count((n + 47) // 48)


def transposed_buffer(rows, cols, device):
    """An empty [cols, rows] bf16 view of a [cols, ceil8(rows)] buffer (the wgrad GEMM wants pitches % 8 == 0)."""
    return torch.empty(cols, (rows + 7) // 8 * 8, dtype=torch.bfloat16, device=device)[:, :rows]


def dropout_add_ln(y, residual=None, gamma=None, beta=None, eps=1e-5, p=0.0, seed=0, site=0, want_x=True):
    """x1 = residual + dropout(y); ln = LayerNorm(x1) in bf16 (when gamma is given).  -> (x1, ln)."""
    lib = _lib.require_device()
    _req(y, torch.float32, "dropout_add_ln.y")
    M, D = y.shape
    if residual is not None:
        _req(residual, torch.float32, "dropout_add_ln.residual")
    x1 = torch.empty_like(y) if want_x else None
    ln = torch.empty(M, D, dtype=torch.bfloat16, device=y.device) if gamma is not None else None
    check(lib.fbkst_dropout_add_ln(y.data_ptr(), _ptr(residual), _ptr(x1), _ptr(ln), _ptr(gamma), _ptr(beta),
                                   float(eps), M, D, float(p), int(seed), int(site), _stream()))
    _count()
    return x1, ln


def ln_bwd(dy, x, gamma, dx=None, eps=1e-5):
    """LayerNorm backward.  dx: fp32 [M, D] holding the residual branch's gradient (accumulated into), or None.
    -> (dx, dgamma [D], dbeta [D])."""
    lib = _lib.require_device()
    _req(dy, torch.float32, "ln_bwd.dy"); _req(x, torch.float32, "ln_bwd.x")
    M, D = x.shape
    acc = 1 if dx is not None else 0
    if dx is None:
        dx = torch.empty_like(x)
    _req(dx, torch.float32, "ln_bwd.dx")
    G = lib.fbkst_ln_bwd_blocks(M)
    partial = torch.empty(G, 2, D, dtype=torch.float32, device=x.device)
    check(lib.fbkst_ln_bwd(dy.data_ptr(), x.data_ptr(), gamma.data_ptr(), dx.data_ptr(), acc, partial.data_ptr(),
                           float(eps), M, D, _stream()))
    dgb = torch.empty(2, D, dtype=torch.float32, device=x.device)
    _count()
    reduce_sum(partial, G, 2 * D, 1, 2 * D, 2 * D, dgb, 2 * D)
    return dx, dgb[0], dgb[1]


def grad_prep(g, act=None, act_scale=1.0, remap=None, want_gb=True, want_gT=True, want_colsum=True, n_pad=None,
              p=0.0, seed=0, site=0, dp_cols=None):
    """See fbkst_grad_prep.  g [M, N] fp32/bf16 (unit column stride).  -> (gb [M, n_pad] bf16 or None,
    gT [N, M] bf16 (a view of a [N, ceil8(M)] buffer) or None, colsum [N] fp32 or None)."""
    lib = _lib.require_device()
    if g.dtype not in (torch.float32, torch.bfloat16, torch.float16) or g.stride(-1) != 1 or g.dim() != 2:
        raise ValueError("fbkst_b200.grad_prep: g must be a 2-D fp32/bf16/fp16 tensor with unit column stride")
    M, N = g.shape
    n_pad = N if n_pad is None else n_pad
    dev = g.device
    if act is not None:
        _req(act, torch.bfloat16, "grad_prep.act")
    gb = torch.empty(M, n_pad, dtype=torch.bfloat16, device=dev) if want_gb else None
    ldt = (M + 7) // 8 * 8
    gT = torch.empty(N, ldt, dtype=torch.bfloat16, device=dev) if want_gT else None
    tiles = (M + 63) // 64
    cs = torch.empty(tiles, n_pad, dtype=torch.float32, device=dev) if want_colsum else None
    inner, outer = remap if remap is not None else (0, 0)
    check(lib.fbkst_grad_prep(g.data_ptr(), {torch.bfloat16: 0, torch.float32: 1, torch.float16: 2}[g.dtype],
                              g.stride(0), _ptr(act),
                              act.stride(0) if act is not None else 0, float(act_scale), inner, outer,
                              _ptr(gb), n_pad, n_pad, _ptr(gT), ldt, _ptr(cs), n_pad, M, N, float(p), int(seed),
                              int(site), int(dp_cols if dp_cols is not None else N), _stream()))
    _count()
    colsum = None
    if want_colsum:
        colsum = torch.empty(n_pad, dtype=torch.float32, device=dev)
        reduce_sum(cs, tiles, n_pad, 1, n_pad, n_pad, colsum, n_pad)
        colsum = colsum[:N]
    return gb, (gT[:, :M] if gT is not None else None), colsum


def transpose_bf16(x):
    """[M, N] bf16/fp32 -> [N, M] bf16 (a view of a [N, ceil8(M)] buffer): the wgrad GEMM's token-contiguous
    operand, or a transposed weight copy for the dgrad GEMM."""
    return grad_prep(x, want_gb=False, want_gT=True, want_colsum=False)[1]


def linear_wgrad(gT, xT):
    """dW [n_out, k_in] fp32 = gT [n_out, tokens] @ xT [k_in, tokens]^T (both bf16, token-contiguous views)."""
    lib = _lib.require_device()
    if gT.dtype != torch.bfloat16 or xT.dtype != torch.bfloat16 or gT.stride(1) != 1 or xT.stride(1) != 1:
        raise ValueError("fbkst_b200.linear_wgrad: operands must be bf16 with unit column stride")
    n_out, tokens = gT.shape
    k_in = xT.shape[0]
    if xT.shape[1] != tokens:
        raise ValueError("fbkst_b200.linear_wgrad: token counts differ")
    ws = torch.empty(lib.fbkst_linear_wgrad_workspace(n_out, k_in, tokens), dtype=torch.float32, device=gT.device)
    dW = torch.empty(n_out, k_in, dtype=torch.float32, device=gT.device)
    # (the reduction of the split-K slices is NOT deferred: run right behind the GEMM it reads the slices from
    # L2; batched at the end of the backward it read 1.9 GB from HBM -- 0.9 ms against 0.45 ms per cfg4 step)
    check(lib.fbkst_linear_wgrad_bf16(gT.data_ptr(), gT.stride(0), xT.data_ptr(), xT.stride(0), ws.data_ptr(),
                                      dW.data_ptr(), k_in, n_out, k_in, tokens, _stream()))
    _count(2)
    return dW


def linear_wgrad_nt(g, x):
    """dW [n_out, k_in] fp32 = g^T x from the natural layouts: g [tokens, n_out] bf16, x [tokens, k_in] bf16
    (unit column strides, pitches % 8 == 0): no transposed copies."""
    lib = _lib.require_device()
    if g.dtype != torch.bfloat16 or x.dtype != torch.bfloat16 or g.stride(1) != 1 or x.stride(1) != 1 or \
            g.shape[0] != x.shape[0]:
        raise ValueError("fbkst_b200.linear_wgrad_nt: g [tokens, n] bf16 and x [tokens, k] bf16 expected")
    tokens, n_out = g.shape
    k_in = x.shape[1]
    ws = torch.empty(lib.fbkst_linear_wgrad_workspace(n_out, k_in, tokens), dtype=torch.float32, device=g.device)
    dW = torch.empty(n_out, k_in, dtype=torch.float32, device=g.device)
    check(lib.fbkst_linear_wgrad_nt(g.data_ptr(), g.stride(0), x.data_ptr(), x.stride(0), 0, ws.data_ptr(),
                                    dW.data_ptr(), k_in, n_out, k_in, tokens, _stream()))
    _count(2)
    return dW


def attention_train_fwd(qkv, lengths, L, B, H, log_penalty=True, p=0.0, seed=0, site=0):
    """Training attention: qkv [L*B, 3*H*64] bf16 UNSCALED -> (out [L*B, H*64] bf16, lse [B*H, L] fp32)."""
    lib = _lib.require_device()
    _req(qkv, torch.bfloat16, "attention_train_fwd.qkv"); _req(lengths, torch.int32, "attention_train_fwd.lengths")
    if qkv.shape != (L * B, 3 * H * 64):
        raise ValueError("fbkst_b200.attention_train_fwd: bad qkv shape %s" % (tuple(qkv.shape),))
    out = torch.empty(L * B, H * 64, dtype=torch.bfloat16, device=qkv.device)
    lse = torch.empty(B * H, L, dtype=torch.float32, device=qkv.device)
    check(lib.fbkst_attention_train_fwd(qkv.data_ptr(), out.data_ptr(), lse.data_ptr(), lengths.data_ptr(), L, B, H,
                                        1 if log_penalty else 0, float(p), int(seed), int(site), _stream()))
    _count()
    return out, lse


def attention_train_bwd(qkv, out, dout, lse, lengths, L, B, H, log_penalty=True, p=0.0, seed=0, site=0):
    """-> dqkv [L*B, 3*H*64] bf16 given dout [L*B, H*64] bf16 (and the forward's out / lse)."""
    lib = _lib.require_device()
    _req(qkv, torch.bfloat16, "attention_train_bwd.qkv"); _req(dout, torch.bfloat16, "attention_train_bwd.dout")
    _req(out, torch.bfloat16, "attention_train_bwd.out"); _req(lse, torch.float32, "attention_train_bwd.lse")
    M = L * B
    delta = torch.empty(M, H, dtype=torch.float32, device=qkv.device)
    check(lib.fbkst_attn_delta(dout.data_ptr(), out.data_ptr(), delta.data_ptr(), M, H, _stream()))
    dqkv = torch.empty(M, 3 * H * 64, dtype=torch.bfloat16, device=qkv.device)
    check(lib.fbkst_attention_train_bwd(qkv.data_ptr(), dout.data_ptr(), lse.data_ptr(), delta.data_ptr(),
                                        dqkv.data_ptr(), lengths.data_ptr(), L, B, H, 1 if log_penalty else 0,
                                        float(p), int(seed), int(site), _stream()))
    _count(3)
    return dqkv


def ctc_compress_bwd(dout, seg_id, weight, L, B):
    lib = _lib.require_device()
    _req(dout, torch.float32, "ctc_compress_bwd.dout")
    D = dout.shape[-1]
    dx = torch.empty(L * B, D, dtype=torch.float32, device=dout.device)
    check(lib.fbkst_ctc_compress_bwd(dout.data_ptr(), seg_id.data_ptr(), weight.data_ptr(), dx.data_ptr(), L, B, D,
                                     _stream()))
    _count()
    return dx


def dropout_(x, p, seed, site):
    """In-place dropout of a contiguous bf16 / fp32 tensor (numel % 4 == 0)."""
    lib = _lib.require_device()
    if p <= 0.0:
        return x
    if x.dtype not in (torch.float32, torch.bfloat16) or not x.is_contiguous():
        raise ValueError("fbkst_b200.dropout_: contiguous bf16/fp32 tensor expected")
    check(lib.fbkst_dropout_inplace(x.data_ptr(), 1 if x.dtype == torch.float32 else 0, x.numel(), float(p),
                                    int(seed), int(site), _stream()))
    _count()
    return x


def bn_batch_stats(y, gamma, beta, eps=1e-5, momentum=0.1, running_mean=None, running_var=None):
    """Training-mode BatchNorm statistics of y [..., C] fp16 (channels-last): -> (mean, rstd, scale, shift) [C]
    fp32; running_mean / running_var (fp32, updated in place) as nn.BatchNorm2d does."""
    lib = _lib.require_device()
    _req(y, torch.float16, "bn_batch_stats.y")
    C = y.shape[-1]
    P = y.numel() // C
    dev = y.device
    out = torch.empty(4, C, dtype=torch.float32, device=dev)
    partial = torch.empty(lib.fbkst_bn_partial_blocks(), 2, C, dtype=torch.float32, device=dev)
    check(lib.fbkst_bn_batch_stats(y.data_ptr(), P, C, gamma.data_ptr(), beta.data_ptr(), float(eps),
                                   float(momentum), _ptr(running_mean), _ptr(running_var), out[0].data_ptr(),
                                   out[1].data_ptr(), out[2].data_ptr(), out[3].data_ptr(), partial.data_ptr(),
                                   _stream()))
    _count(2)
    return out[0], out[1], out[2], out[3]


def bn_apply(x, scale, shift, p=0.0, seed=0, site=0):
    """y = dropout(scale[c] * x + shift[c]); x [..., C] fp16 channels-last -> fp16."""
    lib = _lib.require_device()
    _req(x, torch.float16, "bn_apply.x")
    C = x.shape[-1]
    y = torch.empty_like(x)
    check(lib.fbkst_bn_apply(x.data_ptr(), y.data_ptr(), scale.data_ptr(), shift.data_ptr(), x.numel() // C, C,
                             float(p), int(seed), int(site), _stream()))
    _count()
    return y


def bn_relu_bwd(dy, relu_out, gamma, mean, rstd, batch_stats, p=0.0, seed=0, site=0):
    """-> (dz bf16 like dy, dbeta [C], dgamma [C])."""
    lib = _lib.require_device()
    _req(dy, torch.bfloat16, "bn_relu_bwd.dy"); _req(relu_out, torch.float16, "bn_relu_bwd.relu_out")
    C = dy.shape[-1]
    P = dy.numel() // C
    dz = torch.empty_like(dy)
    sums = torch.empty(2, C, dtype=torch.float32, device=dy.device)
    partial = torch.empty(lib.fbkst_bn_partial_blocks(), 2, C, dtype=torch.float32, device=dy.device)
    check(lib.fbkst_bn_relu_bwd(dy.data_ptr(), relu_out.data_ptr(), gamma.data_ptr(), mean.data_ptr(),
                                rstd.data_ptr(), 1 if batch_stats else 0, dz.data_ptr(), sums.data_ptr(),
                                partial.data_ptr(), P, C, float(p), int(seed), int(site), _stream()))
    _count(3)
    return dz, sums[0], sums[1]


def conv2_im2col_t(y1):
    """y1 [B,T1,F1,C] fp16 -> colT [9*C, B*T2*F2] bf16 (a view of a pitch-padded buffer)."""
    lib = _lib.require_device()
    _req(y1, torch.float16, "conv2_im2col_t.y1")
    B, T1, F1, C = y1.shape
    P2 = B * ((T1 + 1) // 2) * ((F1 + 1) // 2)
    ldt = (P2 + 7) // 8 * 8
    colT = torch.empty(9 * C, ldt, dtype=torch.bfloat16, device=y1.device)
    check(lib.fbkst_conv2_im2col_t(y1.data_ptr(), colT.data_ptr(), ldt, B, T1, F1, C, _stream()))
    _count()
    return colT[:, :P2]


def conv2_col2im(dcol, B, T1, F1, C):
    """dcol [B*T2*F2, 9*C] bf16 -> dy1 [B,T1,F1,C] bf16."""
    lib = _lib.require_device()
    _req(dcol, torch.bfloat16, "conv2_col2im.dcol")
    dy1 = torch.empty(B, T1, F1, C, dtype=torch.bfloat16, device=dcol.device)
    check(lib.fbkst_conv2_col2im(dcol.data_ptr(), dy1.data_ptr(), B, T1, F1, C, _stream()))
    _count()
    return dy1


def conv1_wgrad(dz1, x):
    """dz1 [B,T1,F1,C] bf16, x [B,T,F] fp32 -> (dW1 [C, 9] fp32, db1 [C] fp32)."""
    lib = _lib.require_device()
    _req(dz1, torch.bfloat16, "conv1_wgrad.dz1"); _req(x, torch.float32, "conv1_wgrad.x")
    B, T, Fd = x.shape
    C = dz1.shape[-1]
    out = torch.empty(C, 10, dtype=torch.float32, device=x.device)
    partial = torch.empty(lib.fbkst_bn_partial_blocks(), C, 10, dtype=torch.float32, device=x.device)
    check(lib.fbkst_conv1_wgrad(dz1.data_ptr(), x.data_ptr(), out.data_ptr(), partial.data_ptr(), B, T, Fd, C,
                                _stream()))
    _count(2)
    return out[:, :9], out[:, 9]


def ctc_loss_bwd(logits, lse, in_lengths, targets, target_lengths, blank, grad_loss, L, B, V):
    """d(sum_b nll_b)/d logits * grad_loss -> dlogits [L*B, V] fp32 view of a [L*B, ceil8(V)] buffer."""
    lib = _lib.require_device()
    if logits.dtype not in (torch.bfloat16, torch.float32) or logits.stride(-1) != 1:
        raise ValueError("fbkst_b200.ctc_loss_bwd: logits must be bf16/fp32 with unit column stride")
    _req(lse, torch.float32, "ctc_loss_bwd.lse"); _req(in_lengths, torch.int32, "ctc_loss_bwd.in_lengths")
    _req(target_lengths, torch.int32, "ctc_loss_bwd.target_lengths")
    U = targets.shape[1]
    dev = logits.device
    g = grad_loss.reshape(1).to(torch.float32).contiguous()
    ldd = (V + 7) // 8 * 8
    dz = torch.empty(L * B, ldd, dtype=torch.float32, device=dev)
    ws = torch.empty(max(1, lib.fbkst_ctc_loss_bwd_workspace(L, B, U)), dtype=torch.float32, device=dev)
    check(lib.fbkst_ctc_loss_bwd(logits.data_ptr(), BF16 if logits.dtype == torch.bfloat16 else F32, logits.stride(0),
                                 lse.data_ptr(), in_lengths.data_ptr(), targets.data_ptr() if U else 0,
                                 targets.stride(0) if U else 0, target_lengths.data_ptr(), int(blank), g.data_ptr(),
                                 ws.data_ptr(), dz.data_ptr(), ldd, L, B, V, U, _stream()))
    _count(2)
    return dz[:, :V]
