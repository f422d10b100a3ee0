"""Next row N4 (SURVEY §8f): the decoder's encoder-decoder attention over the compressed encoder
output, and the beam bookkeeping around it, on the sm_100a kernels.

``CrossAttention`` is a drop-in for ``MultiheadAttention(embed_dim, heads, kdim, vdim,
encoder_decoder_attention=True)`` (fairseq/modules/multihead_attention.py:25-83) as
``TransformerDecoderLayer`` calls it (fairseq/modules/transformer_layer.py:339-348): same constructor
arguments, same parameter names (``k_proj / v_proj / q_proj / out_proj`` -> reference checkpoints load
with ``strict=True``), same ``forward`` signature and return values, same incremental-state protocol
(``reorder_incremental_state``, fairseq's ``<uuid>.attn_state`` key).

What changes is the data path:
  * K and V are projected ONCE per utterance into one bf16 buffer ``[S, U, 2D]`` (one tcgen05 GEMM
    with the concatenated k/v weights).  The reference projects the x beam replicated encoder output
    (sequence_generator.py:193-198) and caches ``(bsz*beam, H, S, hd)`` copies per layer (:277-279).
  * every hypothesis row addresses its utterance through ``row_map`` [bsz] int32;
    ``reorder_incremental_state`` gathers that vector instead of ``index_select``-ing the cached K/V
    (:407-420) when finished sentences leave the batch.
  * scores, key-padding mask, fp32 softmax, P.V and the head-averaged weights are one kernel
    (``fbkst_xattn_fwd``); q/out projections are the tcgen05 linear kernel.

``precision = "fp32"`` keeps every operand in fp32 instead: the K/V, q and out projections run on the
split-TF32 GEMM (``ops.linear_f32``) and the core on ``fbkst_xattn_fwd_f32``, the same kernel on fp32
operands; the cached K/V is then ``[S, U, 2D]`` fp32.

The replication is recognised through tags the encoder's ``reorder_encoder_out`` leaves on the tensors
it returns (``beam_source`` below); an untagged ``key`` is simply treated as U = bsz utterances.
There is no CPU / PyTorch fallback, and no backward: training-mode calls with grad enabled raise.
"""
import math
import uuid
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn
from torch import Tensor

from . import ops
from .encoder import PRECISIONS


# ------------------------------------------------------------------ beam tags on encoder outputs
def beam_source(t) -> Tuple[Tensor, Optional[Tensor]]:
    """(base tensor, rows) for a tensor returned by our ``reorder_encoder_out``: ``t`` equals
    ``base.index_select(batch_dim, rows)`` (eager mode, ``_fbkst_src``) or IS the un-replicated base
    carrying the row vector (lazy mode, ``_fbkst_rows``).  Untagged: ``(t, None)``."""
    src = getattr(t, "_fbkst_src", None)
    if src is not None:
        return src
    rows = getattr(t, "_fbkst_rows", None)
    return t, rows


def reorder_tagged(t, batch_dim, new_order, lazy, memo=None):
    """``t.index_select(batch_dim, new_order)`` that remembers where the rows came from.  Chained
    calls compose the index vectors, so the result is always ONE gather from the original encoder
    output.  ``lazy``: do not gather at all -- return an alias of the base tagged with the rows
    (only consumers that understand the tag, i.e. ``CrossAttention``, may read it).  ``memo`` (a dict
    shared by the calls of one ``reorder_encoder_out``) makes tensors that were reordered together
    carry the SAME row-vector object, which is how ``CrossAttention`` recognises that the encoder
    output and its padding mask are replicated identically without comparing device data."""
    base, rows = beam_source(t)
    k = id(rows) if rows is not None else None
    if memo is not None and k in memo:
        rows = memo[k]
    else:
        rows = new_order if rows is None else rows.index_select(0, new_order)
        if memo is not None:
            memo[k] = rows
    if lazy:
        out = base.detach()  # new tensor object, same storage: tags never leak to older tuples
        out._fbkst_rows = rows
        return out
    out = base.index_select(batch_dim, rows)
    out._fbkst_src = (base, rows)
    return out


class CrossAttention(nn.Module):
    def __init__(self, embed_dim, num_heads, kdim=None, vdim=None, dropout=0.0, bias=True,
                 add_bias_kv=False, add_zero_attn=False, self_attention=False,
                 encoder_decoder_attention=True, q_noise=0.0, qn_block_size=8):
        super().__init__()
        if self_attention or not encoder_decoder_attention:
            raise NotImplementedError("fbkst_b200.CrossAttention: encoder-decoder attention only")
        if add_bias_kv or add_zero_attn or q_noise > 0 or not bias:
            raise NotImplementedError("fbkst_b200.CrossAttention: add_bias_kv / add_zero_attn / "
                                      "quant-noise / bias-free projections are not supported")
        self.embed_dim = embed_dim
        self.kdim = kdim if kdim is not None else embed_dim
        self.vdim = vdim if vdim is not None else embed_dim
        if self.kdim != self.vdim:
            raise NotImplementedError("fbkst_b200.CrossAttention: kdim must equal vdim (both are the "
                                      "encoder embedding size in the decoder layer)")
        self.qkv_same_dim = self.kdim == embed_dim and self.vdim == embed_dim
        self.num_heads = num_heads
        self.dropout = dropout
        self.head_dim = embed_dim // num_heads
        if self.head_dim != 64 or self.head_dim * num_heads != embed_dim or num_heads > 16:
            raise NotImplementedError("fbkst_b200.CrossAttention: head_dim must be 64, at most 16 heads")
        self.scaling = self.head_dim ** -0.5
        self.self_attention = False
        self.encoder_decoder_attention = True
        self.k_proj = nn.Linear(self.kdim, embed_dim)
        self.v_proj = nn.Linear(self.vdim, embed_dim)
        self.q_proj = nn.Linear(embed_dim, embed_dim)
        self.out_proj = nn.Linear(embed_dim, embed_dim)
        self.bias_k = self.bias_v = None
        self.add_zero_attn = False
        self.onnx_trace = False
        self.reset_parameters()
        self._incremental_state_id = str(uuid.uuid4())  # incremental_decoding_utils.py:18-19
        self._prep = None
        self._prep_key = None
        self._prep32 = None
        self._prep32_key = None
        self._precision = "bf16"

    @property
    def precision(self):
        """Operand precision of the forward: ``"bf16"`` (default; bf16 tensor-core projections and bf16 K/V,
        q and head outputs) or ``"fp32"`` (split-TF32 projections and an fp32 core: within 1e-3 of an fp32
        reference).  An incremental cache is only valid under the precision it was built with."""
        return self._precision

    @precision.setter
    def precision(self, value):
        if value not in PRECISIONS:
            raise ValueError("fbkst_b200: precision must be one of %s, got %r" % (PRECISIONS, value))
        self._precision = value

    def reset_parameters(self):
        """multihead_attention.py:88-106"""
        if self.qkv_same_dim:
            for m in (self.k_proj, self.v_proj, self.q_proj):
                nn.init.xavier_uniform_(m.weight, gain=1 / math.sqrt(2))
        else:
            for m in (self.k_proj, self.v_proj, self.q_proj):
                nn.init.xavier_uniform_(m.weight)
        nn.init.xavier_uniform_(self.out_proj.weight)
        nn.init.constant_(self.out_proj.bias, 0.0)

    # -------------------------------------------------------------- derived operand formats
    def _params_key(self):
        return tuple((p._version, p.data_ptr()) for p in self.parameters())

    def _prepared(self):
        key = self._params_key()
        if self._prep_key != key:
            with torch.no_grad():
                f = lambda t: t.detach().float().contiguous()
                self._prep = dict(
                    wkv=ops.cast_bf16(torch.cat([f(self.k_proj.weight), f(self.v_proj.weight)], 0)),
                    bkv=torch.cat([f(self.k_proj.bias), f(self.v_proj.bias)], 0),
                    # q *= scaling (:209) folded into the projection: 2^-3, exact in bf16 and fp32
                    wq=ops.cast_bf16(f(self.q_proj.weight), self.scaling),
                    bq=f(self.q_proj.bias) * self.scaling,
                    wo=ops.cast_bf16(f(self.out_proj.weight)), bo=f(self.out_proj.bias))
            self._prep_key = key
        return self._prep

    def _prepared_f32(self):
        key = self._params_key()
        if self._prep32_key != key:
            with torch.no_grad():
                f = lambda t: t.detach().float().contiguous()
                self._prep32 = dict(
                    wkv=torch.cat([f(self.k_proj.weight), f(self.v_proj.weight)], 0),
                    bkv=torch.cat([f(self.k_proj.bias), f(self.v_proj.bias)], 0),
                    wq=f(self.q_proj.weight) * self.scaling, bq=f(self.q_proj.bias) * self.scaling,
                    wo=f(self.out_proj.weight), bo=f(self.out_proj.bias))
            self._prep32_key = key
        return self._prep32

    # ------------------------------------------------------------------ incremental state
    def _full_key(self):
        return "{}.{}".format(self._incremental_state_id, "attn_state")

    def _get_input_buffer(self, incremental_state) -> Dict[str, Optional[Tensor]]:
        if incremental_state is None or self._full_key() not in incremental_state:
            return {}
        return incremental_state[self._full_key()]

    def _set_input_buffer(self, incremental_state, buffer):
        if incremental_state is not None:
            incremental_state[self._full_key()] = buffer
        return incremental_state

    def reorder_incremental_state(self, incremental_state, new_order):
        """multihead_attention.py:407-420.  The reference gathers the cached (bsz, H, S, hd) K/V along
        dim 0 -- unless the cache already has ``new_order``'s batch size, in which case it is left
        alone (hypotheses of one sentence share their K/V).  Same rule here, applied to the row map:
        B*beam int32 values move instead of 2 * bsz * H * S * hd cached elements."""
        buf = self._get_input_buffer(incremental_state)
        rm = buf.get("fbkst_row_map")
        if rm is not None and rm.numel() != new_order.numel():
            buf["fbkst_row_map"] = rm.index_select(0, new_order.to(rm.device))
            self._set_input_buffer(incremental_state, buf)
        return incremental_state

    # ------------------------------------------------------------------------------ forward
    def _project_kv(self, key, key_padding_mask, bsz):
        base, rows = beam_source(key)
        mask = None
        if key_padding_mask is not None:
            mbase, mrows = beam_source(key_padding_mask)
            same = rows is mrows  # both untagged, or reordered together (reorder_tagged's memo)
            if same and mbase.shape[0] == base.shape[1]:
                mask = mbase
            else:  # mask and keys disagree about the replication: fall back to one utterance per row
                base, rows = key, None
                if getattr(key, "_fbkst_rows", None) is not None:
                    raise RuntimeError("fbkst_b200.CrossAttention: lazily reordered encoder output "
                                       "with a key_padding_mask that is not reordered the same way")
                mask = key_padding_mask
        S, U, kd = base.shape
        if kd != self.kdim:
            raise ValueError("fbkst_b200.CrossAttention: key feature size %d != kdim %d" % (kd, self.kdim))
        a = base.reshape(S * U, kd)
        if self._precision == "fp32":
            P = self._prepared_f32()
            kv = ops.linear_f32(a.float().contiguous(), P["wkv"], P["bkv"])
        else:
            P = self._prepared()
            a = ops.cast_bf16(a.float().contiguous()) if a.dtype != torch.bfloat16 else a.contiguous()
            kv = ops.linear(a, P["wkv"], P["bkv"])
        kv = kv.view(S, U, 2 * self.embed_dim)
        if rows is None:
            if U != bsz:
                raise ValueError("fbkst_b200.CrossAttention: %d key columns for %d queries" % (U, bsz))
            row_map = torch.arange(bsz, dtype=torch.int32, device=key.device)
        else:
            row_map = rows.to(device=key.device, dtype=torch.int32)
            if row_map.numel() != bsz:
                raise ValueError("fbkst_b200.CrossAttention: %d tagged rows for %d queries" %
                                 (row_map.numel(), bsz))
        if mask is not None:
            mask = mask.to(torch.bool).contiguous()
        return kv, mask, row_map

    def forward(self, query, key: Optional[Tensor], value: Optional[Tensor],
                key_padding_mask: Optional[Tensor] = None, incremental_state=None,
                need_weights: bool = True, static_kv: bool = False, attn_mask: Optional[Tensor] = None,
                before_softmax: bool = False, need_head_weights: bool = False):
        if self.training and torch.is_grad_enabled():
            raise NotImplementedError("fbkst_b200.CrossAttention: no backward; call eval() / "
                                      "torch.no_grad() (there is no PyTorch fallback)")
        if attn_mask is not None or before_softmax:
            raise NotImplementedError("fbkst_b200.CrossAttention: attn_mask / before_softmax are not "
                                      "part of the encoder-decoder path")
        if not query.is_cuda:
            raise RuntimeError("fbkst_b200.CrossAttention: query must be a CUDA tensor (no CPU fallback)")
        if need_head_weights:
            need_weights = True
        tgt_len, bsz, D = query.shape
        assert D == self.embed_dim
        f32 = self._precision == "fp32"
        with torch.no_grad():
            buf = self._get_input_buffer(incremental_state) if incremental_state is not None else {}
            if "fbkst_kv" in buf and static_kv:  # :181-186: cached, key/value ignored
                kv, mask, row_map = buf["fbkst_kv"], buf["fbkst_mask"], buf["fbkst_row_map"]
                if row_map.numel() != bsz:
                    raise RuntimeError("fbkst_b200.CrossAttention: cached state holds %d hypotheses, "
                                       "query has %d" % (row_map.numel(), bsz))
                # the cached K/V's dtype records the precision it was projected in
                if (kv.dtype == torch.float32) != f32:
                    raise RuntimeError("fbkst_b200.CrossAttention: the incremental state was built with "
                                       "precision=%r, the module now runs precision=%r; start a new "
                                       "incremental state after switching precision" %
                                       ("fp32" if kv.dtype == torch.float32 else "bf16", self._precision))
            else:
                if key is None:
                    raise ValueError("fbkst_b200.CrossAttention: no key and no cached state")
                kv, mask, row_map = self._project_kv(key, key_padding_mask, bsz)
                if incremental_state is not None:
                    self._set_input_buffer(incremental_state, dict(fbkst_kv=kv, fbkst_mask=mask,
                                                                   fbkst_row_map=row_map))
            S, U = kv.shape[0], kv.shape[1]
            qa = query.reshape(tgt_len * bsz, D)
            weights = 2 if need_head_weights else (1 if need_weights else 0)
            if f32:
                P = self._prepared_f32()
                q = ops.linear_f32(qa.float().contiguous(), P["wq"], P["bq"])
                heads, w = ops.xattn_f32(q, kv, mask, row_map, S, U, bsz, tgt_len, self.num_heads, weights)
                attn = ops.linear_f32(heads, P["wo"], P["bo"]).view(tgt_len, bsz, D)
            else:
                P = self._prepared()
                qa = ops.cast_bf16(qa.float().contiguous()) if qa.dtype != torch.bfloat16 else qa.contiguous()
                q = ops.linear(qa, P["wq"], P["bq"])
                if not q.is_contiguous():
                    q = q.contiguous()
                heads, w = ops.xattn(q, kv, mask, row_map, S, U, bsz, tgt_len, self.num_heads, weights=weights)
                attn = ops.linear(heads, P["wo"], P["bo"], out_dtype=torch.float32).view(tgt_len, bsz, D)
            if attn.dtype != query.dtype:
                attn = attn.to(query.dtype)
        return attn, w

    def upgrade_state_dict_named(self, state_dict, name):
        """multihead_attention.py:442-485 splits a legacy fused ``in_proj_weight``; encoder-decoder
        blocks of this reference generation are saved with separate projections already."""
        return state_dict


def swap_cross_attention(decoder, precision="bf16"):
    """Replace every ``layer.encoder_attn`` of a fairseq ``TransformerDecoder`` with a
    ``CrossAttention`` holding the SAME parameter tensors (state_dict keys and values unchanged), and
    set every layer's ``CrossAttention.precision`` (already swapped layers included) to ``precision``.
    Returns the number of layers swapped."""
    if precision not in PRECISIONS:
        raise ValueError("fbkst_b200: precision must be one of %s, got %r" % (PRECISIONS, precision))
    n = 0
    for layer in getattr(decoder, "layers", []):
        old = getattr(layer, "encoder_attn", None)
        if old is None:
            continue
        if isinstance(old, CrossAttention):
            old.precision = precision
            continue
        new = CrossAttention(old.embed_dim, old.num_heads, kdim=old.kdim, vdim=old.vdim,
                             dropout=old.dropout, encoder_decoder_attention=True)
        new.precision = precision
        for nm in ("k_proj", "v_proj", "q_proj", "out_proj"):
            getattr(new, nm).weight = getattr(old, nm).weight
            getattr(new, nm).bias = getattr(old, nm).bias
        layer.encoder_attn = new
        n += 1
    return n
