"""Host-side mirror of the reference's CTC criterion arithmetic (SURVEY §8f N1) over the device path.

Reference: ``examples/speech_recognition/criterions/CTC_loss.py`` -- ``compute_ctc_uer`` (:31-74) and
the ``F.ctc_loss`` call of ``CTCCriterion.forward`` (:128-151), reached from ``ctc_multi_loss.py:27-41``
with the encoder's ``ctc_out`` (T x B x V) and ``ctc_padding_mask``.

The reference pulls every utterance's arg-max path to the host (``.tolist()``), collapses it with
``itertools.groupby`` and runs a Python O(P*U) alignment per utterance, every training and validation
step.  Here the frame arg-max, the log-sum-exp, the collapse, the alignment and the alpha recursion
all run on the GPU; the only host transfer is the final read of 3 scalars.

No CPU fallback: CPU tensors raise.
"""
from typing import Callable, NamedTuple, Optional

import torch

from . import ops


def _time_major_rows(x):
    """[T, B, V] logits/log-probs -> ([T*B, V] row view with row t*B+b, T, B, V) without copying
    when the storage is time-major (also when `x` is the criterion's N x T x D transposed view)."""
    if x.dim() != 3:
        raise ValueError("fbkst_b200.criterion: expected a 3-D tensor")
    if not x.is_cuda:
        raise ValueError("fbkst_b200.criterion: expected a CUDA tensor (there is no CPU fallback)")
    if x.dtype not in (torch.bfloat16, torch.float32):
        x = x.float()
    T, B, V = x.shape
    if x.stride(2) != 1 or x.stride(0) != B * x.stride(1):
        x = x.contiguous()
    return x.as_strided((T * B, V), (x.stride(1), 1), x.storage_offset()), T, B, V


def _i32(t, device):
    return torch.as_tensor(t, device=device).to(torch.int32).contiguous()


def ctc_uer_device(ctc_out, targets, input_lengths, target_lengths, blank_idx):
    """Device tensors only, no synchronisation.  ctc_out T x B x V (logits or log-probs: the arg-max
    is the same).  -> (errors [B] int32, totals [2] int64 = (batch_errors, batch_total))."""
    rows, T, B, V = _time_major_rows(ctc_out)
    dev = rows.device
    il, tl = _i32(input_lengths, dev), _i32(target_lengths, dev)
    labels, _ = ops.ctc_argmax(rows, il, T, B, V, want_prob=False)
    tg = torch.as_tensor(targets, device=dev).to(torch.int64)
    errors, _, totals = ops.ctc_uer(labels, il, tg, tl, blank_idx, T, B)
    return errors, totals


def compute_ctc_uer(logprobs, targets, input_lengths, target_lengths, blank_idx):
    """Same signature and return value as the reference's ``compute_ctc_uer`` (CTC_loss.py:31-74):
    logprobs N x T1 x D (the criterion passes the transposed view of the T x N x D tensor, which is
    consumed without a copy), targets N x T2, lengths per sample.  Returns (batch_errors, batch_total)
    as Python numbers (one device->host read of 16 bytes)."""
    _, totals = ctc_uer_device(logprobs.transpose(0, 1), targets, input_lengths, target_lengths, blank_idx)
    e, n = totals.tolist()
    return float(e), float(n)


class CtcLossFn(torch.autograd.Function):
    """sum_b nll_b of F.ctc_loss(log_softmax(logits), ..., reduction="sum", zero_infinity=True), differentiable
    w.r.t. the logits on the device kernels (alpha pass forward; dense softmax term + alpha/beta occupancies
    backward).  The log-probabilities are never materialised (the reference's autograd keeps a T x B x V
    log_softmax output alive for the backward)."""

    @staticmethod
    def forward(ctx, ctc_out, in_lengths, targets, target_lengths, blank_idx):
        rows, T, B, V = _time_major_rows(ctc_out)
        labels, lse, _ = ops.ctc_argmax_lse(rows, in_lengths, T, B, V)
        nll, loss = ops.ctc_loss_fwd(rows, lse, in_lengths, targets, target_lengths, blank_idx, T, B, V)
        ctx.save_for_backward(rows, lse, in_lengths, targets, target_lengths)
        ctx.dims = (T, B, V, blank_idx, tuple(ctc_out.shape))
        ctx.mark_non_differentiable(labels, nll)
        return loss.reshape(()), labels, nll

    @staticmethod
    def backward(ctx, grad_loss, _gl, _gn):
        rows, lse, il, tg, tl = ctx.saved_tensors
        T, B, V, blank, shape = ctx.dims
        dz = ops.ctc_loss_bwd(rows, lse, il, tg, tl, blank, grad_loss, T, B, V)  # [T*B, V], pitch ceil8(V)
        return dz.view(T, B, V), None, None, None, None


class Projection(NamedTuple):
    """A CTC projection logits = x W^T + b as the loss node sees it: the parameters, the bf16 transposed weight
    ``weight_t()`` (a [D, V] view of a [D, ceil8(V)] buffer whose pad columns are zero: the dgrad GEMM contracts
    over the padded V) and the encoder whose pending activation transposes its backward starts (or None)."""
    weight: torch.Tensor
    bias: Optional[torch.Tensor]
    weight_t: Callable[[], torch.Tensor]
    encoder: object


def _encoder_projection(enc):
    """The encoder's own ``ctc_fc`` (--ctc-compress-out), operands from its training weight copies."""
    from .train import prepare_train_weights
    return Projection(enc.ctc_fc.weight, enc.ctc_fc.bias, lambda: prepare_train_weights(enc)["wcT"], enc)


def _bf16_rows(x):
    """bf16 GEMM operand copy of [M, D] rows held in fp32, fp16 (model.half()) or bf16."""
    if x.dtype == torch.float32:
        return ops.cast_bf16(x)
    if x.dtype == torch.bfloat16:
        return x.contiguous()
    return ops.grad_prep(x.contiguous(), want_gT=False, want_colsum=False)[0]


def _as(t, like):
    return t if like is None or t is None or t.dtype == like.dtype else t.to(like.dtype)


def _projection_backward(dz, xb, wT, want_dw=True):
    """The projection's backward from d logits ``dz`` [M, V] (unit column stride), the bf16 input rows ``xb``
    [M, D] and the transposed weight ``wT`` (``Projection.weight_t``; None: no dx): -> (dx [M, D] fp32,
    dW [V, D] fp32, db [V] fp32); the parts not wanted are None."""
    M, V = dz.shape
    D = xb.shape[1]
    Vp = (V + 7) // 8 * 8
    gb, gT, dbias = ops.grad_prep(dz, n_pad=Vp, want_gb=wT is not None, want_gT=want_dw, want_colsum=want_dw)
    dW = ops.linear_wgrad(gT, ops.transpose_bf16(xb)) if want_dw else None
    dx = None
    if wT is not None:
        wT_full = wT if Vp == V else torch.as_strided(wT, (D, Vp), (wT.stride(0), 1))
        dx = ops.linear(gb, wT_full, None, out_dtype=torch.float32)
    return dx, dW, dbias


class CtcProjLossFn(torch.autograd.Function):
    """``CtcLossFn`` + the backward of the CTC projection in ONE node: the encoder's ``ctc_fc``
    (conv_transformer.py:278-280) or the criterion's own ``fc_out`` on an intermediate state (``CtcProjection``).

    Why: autograd runs nodes in reverse creation order, so the loss nodes run first, then the whole decoder
    backward (bound by the host's launch rate, GPU nearly idle), and only then the encoder's node.  With the
    projection's backward here -- d logits, d W_ctc = d logits^T x, d b_ctc, d x = d logits W_ctc, the largest
    GEMMs of the step (V = 8005) -- that work executes on the GPU WHILE the host walks the decoder's backward
    instead of on the GPU-bound stretch after it.  ``x`` is the projection's input handed out as a tap
    (``ctc_out._fbkst_tap``); ``logits`` are the values (already computed, hooks applied); ``proj`` is a
    ``Projection``."""

    @staticmethod
    def forward(ctx, logits, x, weight, bias, proj, in_lengths, targets, target_lengths, blank_idx):
        rows, T, B, V = _time_major_rows(logits)
        labels, lse, _ = ops.ctc_argmax_lse(rows, in_lengths, T, B, V)
        nll, loss = ops.ctc_loss_fwd(rows, lse, in_lengths, targets, target_lengths, blank_idx, T, B, V)
        ctx.save_for_backward(rows, lse, in_lengths, targets, target_lengths, x)
        ctx.dims = (T, B, V, blank_idx)
        ctx.proj = proj
        ctx.mark_non_differentiable(labels, nll)
        return loss.reshape(()), labels, nll

    @staticmethod
    def backward(ctx, grad_loss, _gl, _gn):
        from .train import pretranspose
        rows, lse, il, tg, tl, x = ctx.saved_tensors
        T, B, V, blank = ctx.dims
        proj = ctx.proj
        enc = proj.encoder
        if enc is not None:
            # this node runs FIRST in the backward: enqueue the encoder's activation transposes now, so that they
            # execute while the host walks the decoder's backward
            pretranspose(getattr(enc, "_train_pending", None))
            enc._train_pending = None
        wT = proj.weight_t()
        D = x.shape[-1]
        dz = ops.ctc_loss_bwd(rows, lse, il, tg, tl, blank, grad_loss, T, B, V)  # [M, V] fp32, pitch ceil8(V)
        dx, dW, dbias = _projection_backward(dz, _bf16_rows(x.reshape(T * B, D)), wT)
        return (None, _as(dx.view(x.shape), x), _as(dW, proj.weight), _as(dbias, proj.bias),
                None, None, None, None, None)


class _CtcProjectionFn(torch.autograd.Function):
    """The projection as its own autograd node (the route when nothing fuses it with the loss): tcgen05 GEMMs
    forward (logits = bf16(x) W^T + b, fp32) and backward (``_projection_backward``)."""

    @staticmethod
    def forward(ctx, x, weight, bias, mod):
        w, _, b = mod.operands()
        D = x.shape[-1]
        xb = _bf16_rows(x.reshape(-1, D))
        logits = ops.linear(xb, w, b, out_dtype=torch.float32)  # [M, V] view, padded row pitch
        ctx.save_for_backward(xb)
        ctx.mod, ctx.x_meta = mod, (x.shape, x.dtype)
        return logits.view(*x.shape[:-1], logits.shape[1])

    @staticmethod
    def backward(ctx, dy):
        if dy is None:
            return None, None, None, None
        (xb,) = ctx.saved_tensors
        mod = ctx.mod
        shape, dtype = ctx.x_meta
        V = dy.shape[-1]
        dz = dy.reshape(-1, V)
        if dz.stride(-1) != 1:
            dz = dz.contiguous()
        want_dx = ctx.needs_input_grad[0]
        want_dw = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        dx, dW, dbias = _projection_backward(dz, xb, mod.operands()[1] if want_dx else None, want_dw)
        dx = dx.view(shape).to(dtype) if dx is not None else None
        return (dx, _as(dW, mod.weight) if ctx.needs_input_grad[1] else None,
                _as(dbias, mod.bias) if ctx.needs_input_grad[2] else None, None)


class CtcProjection(torch.nn.Module):
    """A CTC projection ``nn.Linear`` (the criterion's own ``fc_out`` of the CTC-multitask recipe without
    --ctc-compress-out: ctc_multi_loss projects ``encoder_states[ctc_encoder_layer - 1]`` with it) on the tcgen05
    GEMM.  Holds the SAME Parameter objects as the Linear it wraps (state-dict keys, optimizer state and
    fairseq's fp16 master copies are unchanged); bf16 operand copies are re-derived whenever a parameter's
    version counter or storage changes (after every optimizer step, ``.half()``, ``.cuda()``).

    forward(x [..., D] fp32 / fp16 / bf16) -> fp32 logits [..., V] (a view with a padded row pitch, as the
    encoder's ``ctc_out``).  With gradients enabled the output carries ``_fbkst_tap = (x, self)``: handed to
    ``ctc_loss_train`` unchanged, the projection's backward runs inside the loss node (``CtcProjLossFn``);
    otherwise its own autograd node computes it.  Under ``no_grad`` it is a plain forward."""

    def __init__(self, linear):
        super().__init__()
        if not isinstance(linear, torch.nn.Linear):
            raise TypeError("CtcProjection wraps an nn.Linear, got %s" % type(linear).__name__)
        self.in_features, self.out_features = linear.in_features, linear.out_features
        self.weight = linear.weight
        self.bias = linear.bias
        self._ops_key, self._ops = None, None

    def extra_repr(self):
        return "in_features=%d, out_features=%d, bias=%s" % (self.in_features, self.out_features,
                                                            self.bias is not None)

    def operands(self):
        """(W [V, D] bf16, W^T [D, V] bf16 view of a [D, ceil8(V)] buffer with zero pad columns, bias fp32)."""
        w, b = self.weight, self.bias
        key = (w._version, w.data_ptr(), w.dtype) + ((b._version, b.data_ptr()) if b is not None else ())
        if self._ops_key == key:
            return self._ops
        if not w.is_cuda:
            raise ValueError("fbkst_b200.CtcProjection: CUDA parameters expected (there is no CPU fallback)")
        V, D = w.shape
        with torch.no_grad():
            old = self._ops
            if old is None or old[0].device != w.device:
                wc = torch.empty(V, D, dtype=torch.bfloat16, device=w.device)
                wT = torch.zeros(D, (V + 7) // 8 * 8, dtype=torch.bfloat16, device=w.device)[:, :V]
            else:
                wc, wT = old[0], old[1]
            src = w.detach()
            ops.prep_batch([(src if src.stride(1) == 1 else src.contiguous(), wc, wT)])
            bc = b.detach().float().contiguous() if b is not None else None
        self._ops, self._ops_key = (wc, wT, bc), key
        return self._ops

    def projection(self, x):
        """This module as the ``Projection`` the fused loss node reads, for the input ``x``."""
        return Projection(self.weight, self.bias, lambda: self.operands()[1], getattr(x, "_fbkst_encoder", None))

    def forward(self, x):
        if not x.is_cuda:
            raise ValueError("fbkst_b200.CtcProjection: expected a CUDA tensor (there is no CPU fallback)")
        if x.shape[-1] != self.in_features:
            raise ValueError("fbkst_b200.CtcProjection: input has %d features, expected %d"
                             % (x.shape[-1], self.in_features))
        if not torch.is_grad_enabled():
            w, _, b = self.operands()
            D = x.shape[-1]
            logits = ops.linear(_bf16_rows(x.reshape(-1, D)), w, b, out_dtype=torch.float32)
            return logits.view(*x.shape[:-1], logits.shape[1])
        y = _CtcProjectionFn.apply(x, self.weight, self.bias, self)
        if y.requires_grad:
            y._fbkst_tap = (x, self)
        return y


def find_ctc_projection(module):
    """-> (parent module, attribute name, module) of the single ``nn.Linear`` (or an installed ``CtcProjection``)
    under ``module`` whose name ends in ``fc_out``: the CTC-multitask criterion's projection
    (``ctc_aware_model.fc_out``; the reference model's raw_state_dict_upgrade moves its weights into
    ``encoder.ctc_fc``).
    Raises ValueError unless there is exactly one."""
    hits = [(n, m) for n, m in module.named_modules()
            if n.split(".")[-1].endswith("fc_out") and isinstance(m, (torch.nn.Linear, CtcProjection))]
    if len(hits) != 1:
        raise ValueError("fbkst_b200: expected exactly one nn.Linear named '*fc_out' in the CTC criterion (its CTC "
                         "projection), found %d: %s" % (len(hits), [n for n, _ in hits]))
    name, mod = hits[0]
    parent = module.get_submodule(name.rsplit(".", 1)[0]) if "." in name else module
    return parent, name.split(".")[-1], mod


def install_ctc_projection(module):
    """Swap the criterion's CTC projection (``find_ctc_projection``) for a ``CtcProjection`` holding the same
    parameters.  Idempotent.  -> the ``CtcProjection``."""
    parent, attr, mod = find_ctc_projection(module)
    if isinstance(mod, CtcProjection):
        return mod
    proj = CtcProjection(mod)
    setattr(parent, attr, proj)
    return proj


def ctc_loss_and_uer(ctc_out, ctc_padding_mask, targets, target_lengths, blank_idx, pad_idx=None):
    """What ``CTCCriterion.forward`` computes from the encoder output (CTC_loss.py:118-154):

        lprobs = log_softmax(ctc_out.float());  input_lengths from the padding mask
        loss   = F.ctc_loss(lprobs, targets, input_lengths, target_lengths, blank, "sum", zero_infinity)
        errors, total = compute_ctc_uer(lprobs, targets, input_lengths, target_lengths, blank)

    ctc_out T x B x V (bf16 or fp32 logits, ``encoder_out.ctc_out``), ctc_padding_mask B x T bool
    (True = padding) or None or a [B] tensor of lengths.  One pass over the logits produces the frame
    arg-max and the log-sum-exp; the log-probabilities are never materialised.
    Returns device tensors (loss [1] fp32, nll [B] fp32, errors [B] int32, totals [2] int64)."""
    rows, T, B, V = _time_major_rows(ctc_out)
    dev = rows.device
    if ctc_padding_mask is None:
        il = torch.full((B,), T, dtype=torch.int32, device=dev)
    elif ctc_padding_mask.dim() == 1:
        il = _i32(ctc_padding_mask, dev)
    else:  # data_utils.encoder_padding_mask_to_lengths: T - number of padded positions
        m = ctc_padding_mask if ctc_padding_mask.shape[0] == B else ctc_padding_mask.t()
        il = (T - m.sum(dim=1)).to(torch.int32)
    tl = _i32(target_lengths, dev)
    tg = torch.as_tensor(targets, device=dev).to(torch.int64)
    labels, lse, _ = ops.ctc_argmax_lse(rows, il, T, B, V)
    nll, loss = ops.ctc_loss_fwd(rows, lse, il, tg, tl, blank_idx, T, B, V)
    errors, _, totals = ops.ctc_uer(labels, il, tg, tl, blank_idx, T, B)
    return loss, nll, errors, totals


def ctc_loss_train(ctc_out, ctc_padding_mask, targets, target_lengths, blank_idx, mask_time_first=True):
    """Differentiable CTC loss + UER counts for the training criterion.  ctc_out T x B x V logits (attached to
    the autograd graph), ctc_padding_mask bool (True = padding), T x B if ``mask_time_first`` (what
    CTCEncoderWrapperModel hands over, ctc_multi_loss.py:41) else B x T, or None.
    -> (loss 0-dim tensor with grad_fn, errors total (device int64 [2]), input_lengths int32 [B])."""
    T, B, V = ctc_out.shape
    dev = ctc_out.device
    if ctc_padding_mask is None:
        il = torch.full((B,), T, dtype=torch.int32, device=dev)
    else:
        il = (T - ctc_padding_mask.sum(dim=0 if mask_time_first else 1)).to(torch.int32)
    tl = _i32(target_lengths, dev)
    tg = torch.as_tensor(targets, device=dev).to(torch.int64).contiguous()
    tap = getattr(ctc_out, "_fbkst_tap", None)
    proj = None
    if tap is not None:
        # the encoder's own training forward (ctc_fc) or a CtcProjection produced these logits: the projection's
        # backward is done in the loss node
        x, owner = tap
        proj = owner.projection(x) if isinstance(owner, CtcProjection) else _encoder_projection(owner)
    if proj is not None and x.requires_grad and proj.weight.requires_grad:
        loss, labels, _ = CtcProjLossFn.apply(ctc_out.detach(), x, proj.weight, proj.bias, proj, il, tg, tl,
                                              int(blank_idx))
    else:
        loss, labels, _ = CtcLossFn.apply(ctc_out, il, tg, tl, int(blank_idx))
    _, _, totals = ops.ctc_uer(labels, il, tg, tl, blank_idx, T, B)
    return loss, totals, il
