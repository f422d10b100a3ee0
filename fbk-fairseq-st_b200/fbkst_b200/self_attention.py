"""Next row N5: the decoder's self-attention during generation on the sm_100a kernels, with an append-only
K/V cache that beam reorders never copy.

``DecoderSelfAttention`` is a drop-in for ``MultiheadAttention(embed_dim, heads, dropout=...,
self_attention=True)`` (fairseq/modules/multihead_attention.py:25-83) as ``TransformerDecoderLayer`` uses it:
same constructor arguments, same parameter names (``k_proj / v_proj / q_proj / out_proj`` -> reference
checkpoints load with ``strict=True``), same ``forward`` signature and return values, same incremental-state
protocol (``_get_input_buffer`` / ``_set_input_buffer``, ``reorder_incremental_state``, fairseq's
``<uuid>.attn_state`` key).

What changes is the data path of incremental decoding.  The reference appends every step's key and value to
per-hypothesis ``(bsz, H, t, 64)`` caches with ``torch.cat`` (a new copy of the whole cache per layer and step)
and ``index_select``s the whole cache again in ``reorder_incremental_state`` (:407-420).  Here:
  * one GEMM per step with ``[W_q * 2^-3; W_k; W_v]`` writes the step's q, k and v of every live hypothesis
    straight into slab t of the layer's cache ``[T_cap, R, 3D]`` (R = hypothesis count at the first step);
    nothing else ever writes or copies that slab;
  * the incremental state holds the cache, the int32 ancestry table ``anc [T_cap, bsz]`` (``anc[s, b]`` is the
    cache row that holds, at step s, the ancestor of hypothesis b), the step count (a host int) and the optional
    key-padding bytes ``[T_cap, R]``, which like K/V are indexed by (step, cache row);
  * ``reorder_incremental_state`` is ``anc = anc.index_select(1, new_order)`` and nothing else -- same-size
    beam permutations and a batch that shrinks as sentences finish alike; the kernel
    (``fbkst_dec_self_attn_fwd``) gathers the keys and values through ``anc``;
  * ``T_cap`` grows geometrically (doubling from ``INITIAL_STEPS``): one copy of the cache per doubling, not
    per step.

``precision = "fp32"`` keeps every operand in fp32: the projections run on the split-TF32 GEMM and the core on
``fbkst_dec_self_attn_fwd_f32``; the cache is then fp32.  The cache's dtype records the precision it was built
with, so a cached step under the other precision raises.

Without an incremental state (``SequenceScorer``, ``--score-reference``) the whole target is projected at once
and attended under fairseq's future mask or no mask.  There is no CPU / PyTorch fallback, and no backward:
training-mode calls with grad enabled raise.
"""
import uuid
from typing import Optional

import torch
import torch.nn as nn
from torch import Tensor

from . import ops
from .cross_attention import CrossAttention
from .encoder import PRECISIONS


class DecoderSelfAttention(nn.Module):
    INITIAL_STEPS = 32  # cache capacity of a new incremental state, in decoder steps

    def __init__(self, embed_dim, num_heads, kdim=None, vdim=None, dropout=0.0, bias=True,
                 add_bias_kv=False, add_zero_attn=False, self_attention=True,
                 encoder_decoder_attention=False, q_noise=0.0, qn_block_size=8):
        super().__init__()
        if not self_attention or encoder_decoder_attention:
            raise NotImplementedError("fbkst_b200.DecoderSelfAttention: self-attention only (use CrossAttention "
                                      "for encoder-decoder attention)")
        if add_bias_kv or add_zero_attn or q_noise > 0 or not bias:
            raise NotImplementedError("fbkst_b200.DecoderSelfAttention: add_bias_kv / add_zero_attn / "
                                      "quant-noise / bias-free projections are not supported")
        if kdim not in (None, embed_dim) or vdim not in (None, embed_dim):
            raise NotImplementedError("fbkst_b200.DecoderSelfAttention: kdim and vdim must equal embed_dim")
        self.embed_dim = embed_dim
        self.kdim = self.vdim = embed_dim
        self.qkv_same_dim = True
        self.num_heads = num_heads
        self.dropout = dropout
        self.head_dim = embed_dim // num_heads
        if self.head_dim != 64 or self.head_dim * num_heads != embed_dim or num_heads > 16:
            raise NotImplementedError("fbkst_b200.DecoderSelfAttention: head_dim must be 64, at most 16 heads")
        self.scaling = self.head_dim ** -0.5
        self.self_attention = True
        self.encoder_decoder_attention = False
        self.k_proj = nn.Linear(embed_dim, embed_dim)
        self.v_proj = nn.Linear(embed_dim, embed_dim)
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

    # the precision switch, parameter init and incremental-state keying are CrossAttention's
    precision = CrossAttention.precision
    reset_parameters = CrossAttention.reset_parameters
    _params_key = CrossAttention._params_key
    _full_key = CrossAttention._full_key
    _get_input_buffer = CrossAttention._get_input_buffer
    _set_input_buffer = CrossAttention._set_input_buffer

    # -------------------------------------------------------------- derived operand formats
    def _qkv_f32(self):
        f = lambda t: t.detach().float().contiguous()
        # q *= scaling (:209) folded into the projection: 2^-3, exact in bf16 and fp32
        w = torch.cat([f(self.q_proj.weight) * self.scaling, f(self.k_proj.weight), f(self.v_proj.weight)], 0)
        b = torch.cat([f(self.q_proj.bias) * self.scaling, f(self.k_proj.bias), f(self.v_proj.bias)], 0)
        return w, b, f(self.out_proj.weight), f(self.out_proj.bias)

    def _prepared(self):
        key = self._params_key()
        if self._prep_key != key:
            with torch.no_grad():
                w, b, wo, bo = self._qkv_f32()
                self._prep = dict(wqkv=ops.cast_bf16(w), bqkv=b, wo=ops.cast_bf16(wo), bo=bo)
            self._prep_key = key
        return self._prep

    def _prepared_f32(self):
        key = self._params_key()
        if self._prep32_key != key:
            with torch.no_grad():
                w, b, wo, bo = self._qkv_f32()
                self._prep32 = dict(wqkv=w, bqkv=b, wo=wo, bo=bo)
            self._prep32_key = key
        return self._prep32

    # ------------------------------------------------------------------ incremental state
    def reorder_incremental_state(self, incremental_state, new_order):
        """multihead_attention.py:407-420 gathers every cached K/V (and padding) tensor along the hypothesis
        dimension.  Here only the ancestry table moves: ``anc.index_select(1, new_order)``, bsz * T_cap int32
        values.  The cache and its padding bytes are indexed by cache row and are never touched."""
        buf = self._get_input_buffer(incremental_state)
        anc = buf.get("fbkst_anc")
        if anc is not None:
            buf["fbkst_anc"] = anc.index_select(1, new_order.to(anc.device))
            self._set_input_buffer(incremental_state, buf)
        return incremental_state

    # ------------------------------------------------------------------------------ forward
    def _project(self, x, out, P, f32):
        """q | k | v of the rows of ``x`` straight into ``out`` (a [rows, 3D] view with any row pitch)."""
        if f32:
            ops.linear_f32(x, P["wqkv"], P["bqkv"], out=out)
        else:
            ops.linear(x, P["wqkv"], P["bqkv"], out=out)

    def _step(self, x, key_padding_mask, incremental_state, bsz, P, f32, weights):
        D, dev = self.embed_dim, x.device
        buf = self._get_input_buffer(incremental_state)
        cache = buf.get("fbkst_cache")
        if cache is None:
            t, pad = 0, None
            cache = torch.empty(self.INITIAL_STEPS, bsz, 3 * D, dtype=torch.float32 if f32 else torch.bfloat16,
                                device=dev)
            anc = torch.empty(self.INITIAL_STEPS, bsz, dtype=torch.int32, device=dev)
        else:
            # the cache's dtype records the precision it was projected in
            if (cache.dtype == torch.float32) != f32:
                raise RuntimeError("fbkst_b200.DecoderSelfAttention: the incremental state was built with "
                                   "precision=%r, the module now runs precision=%r; start a new incremental "
                                   "state after switching precision" %
                                   ("fp32" if cache.dtype == torch.float32 else "bf16", self._precision))
            anc, pad, t = buf["fbkst_anc"], buf["fbkst_pad"], buf["fbkst_steps"]
            if anc.shape[1] != bsz:
                raise RuntimeError("fbkst_b200.DecoderSelfAttention: cached state holds %d hypotheses, query has "
                                   "%d" % (anc.shape[1], bsz))
            if t == cache.shape[0]:  # full: double the capacity (the only copy of the cache)
                grown = cache.new_empty((2 * t,) + tuple(cache.shape[1:]))
                grown[:t] = cache
                cache = grown
                grown = anc.new_empty(2 * t, bsz)
                grown[:t] = anc
                anc = grown
                if pad is not None:
                    grown = pad.new_zeros(2 * t, pad.shape[1])
                    grown[:t] = pad
                    pad = grown
        if key_padding_mask is not None:
            if tuple(key_padding_mask.shape) != (bsz, 1):
                raise ValueError("fbkst_b200.DecoderSelfAttention: an incremental step takes the current "
                                 "token's key_padding_mask [bsz, 1], got %s" % (tuple(key_padding_mask.shape),))
            if pad is None:  # earlier steps had no padding
                pad = torch.zeros(cache.shape[:2], dtype=torch.uint8, device=dev)
            pad[t, :bsz] = key_padding_mask[:, 0]
        torch.arange(bsz, out=anc[t])  # each hypothesis wrote its own row of slab t
        self._project(x, cache[t, :bsz], P, f32)
        fn = ops.dec_self_attn_f32 if f32 else ops.dec_self_attn
        heads, w = fn(cache[t, :bsz, :D], cache, anc, pad, t + 1, bsz, 1, self.num_heads,
                      mode=ops.SA_INCREMENTAL, weights=weights)
        buf.update(fbkst_cache=cache, fbkst_anc=anc, fbkst_pad=pad, fbkst_steps=t + 1)
        self._set_input_buffer(incremental_state, buf)
        return heads, w

    def _full(self, x, key_padding_mask, attn_mask, tgt_len, bsz, P, f32, weights):
        D = self.embed_dim
        mode = ops.SA_FULL
        if attn_mask is not None:
            future = torch.triu(torch.full((tgt_len, tgt_len), float("-inf"), device=attn_mask.device), 1)
            if tuple(attn_mask.shape) != (tgt_len, tgt_len) or not torch.equal(attn_mask.float(), future):
                raise NotImplementedError("fbkst_b200.DecoderSelfAttention: attn_mask must be None or fairseq's "
                                          "future mask (-inf strictly above the diagonal, 0 elsewhere)")
            mode = ops.SA_CAUSAL
        pad = None
        if key_padding_mask is not None:
            if tuple(key_padding_mask.shape) != (bsz, tgt_len):
                raise ValueError("fbkst_b200.DecoderSelfAttention: key_padding_mask must be [bsz, tgt_len] = %s, "
                                 "got %s" % ((bsz, tgt_len), tuple(key_padding_mask.shape)))
            pad = key_padding_mask.t().to(device=x.device, dtype=torch.uint8).contiguous()  # [step, row]
        cache = torch.empty(tgt_len, bsz, 3 * D, dtype=x.dtype, device=x.device)
        self._project(x, cache.view(tgt_len * bsz, 3 * D), P, f32)
        fn = ops.dec_self_attn_f32 if f32 else ops.dec_self_attn
        return fn(cache.view(tgt_len * bsz, 3 * D)[:, :D], cache, None, pad, tgt_len, bsz, tgt_len, self.num_heads,
                  mode=mode, weights=weights)

    def forward(self, query, key: Optional[Tensor], value: Optional[Tensor],
                key_padding_mask: Optional[Tensor] = None, incremental_state=None,
                need_weights: bool = True, static_kv: bool = False, attn_mask: Optional[Tensor] = None,
                before_softmax: bool = False, need_head_weights: bool = False):
        """As ``MultiheadAttention.forward`` with ``self_attention=True``: ``key`` and ``value`` are ignored
        (the layer passes the query).  With ``incremental_state``: one new token per hypothesis (``tgt_len`` 1),
        no ``attn_mask``, ``key_padding_mask`` [bsz, 1] for that token.  Without: ``attn_mask`` None or the
        future mask, ``key_padding_mask`` [bsz, tgt_len].  A query whose keys are all padding gets a zero
        attention row (the reference would produce NaN)."""
        if self.training and torch.is_grad_enabled():
            raise NotImplementedError("fbkst_b200.DecoderSelfAttention: no backward; call eval() / "
                                      "torch.no_grad() (there is no PyTorch fallback)")
        if before_softmax or static_kv:
            raise NotImplementedError("fbkst_b200.DecoderSelfAttention: before_softmax / static_kv are not "
                                      "part of the decoder self-attention path")
        if not query.is_cuda:
            raise RuntimeError("fbkst_b200.DecoderSelfAttention: query must be a CUDA tensor (no CPU fallback)")
        if need_head_weights:
            need_weights = True
        tgt_len, bsz, D = query.shape
        if D != self.embed_dim:
            raise ValueError("fbkst_b200.DecoderSelfAttention: query feature size %d != embed_dim %d" %
                             (D, self.embed_dim))
        f32 = self._precision == "fp32"
        weights = 2 if need_head_weights else (1 if need_weights else 0)
        with torch.no_grad():
            x = query.reshape(tgt_len * bsz, D)
            if f32:
                P = self._prepared_f32()
                x = x.float().contiguous()
            else:
                P = self._prepared()
                x = ops.cast_bf16(x.float().contiguous()) if x.dtype != torch.bfloat16 else x.contiguous()
            if incremental_state is not None:
                if tgt_len != 1 or attn_mask is not None:
                    raise NotImplementedError("fbkst_b200.DecoderSelfAttention: an incremental step takes one "
                                              "token per hypothesis and no attn_mask")
                heads, w = self._step(x, key_padding_mask, incremental_state, bsz, P, f32, weights)
            else:
                heads, w = self._full(x, key_padding_mask, attn_mask, tgt_len, bsz, P, f32, weights)
            if f32:
                attn = ops.linear_f32(heads, P["wo"], P["bo"])
            else:
                attn = ops.linear(heads, P["wo"], P["bo"], out_dtype=torch.float32)
            attn = attn.view(tgt_len, bsz, D)
            if attn.dtype != query.dtype:
                attn = attn.to(query.dtype)
        return attn, w

    def upgrade_state_dict_named(self, state_dict, name):
        """multihead_attention.py:442-485 splits a legacy fused ``in_proj_weight``; decoder blocks of this
        reference generation are saved with separate projections already."""
        return state_dict


def swap_self_attention(decoder, precision="bf16"):
    """Replace every ``layer.self_attn`` of a fairseq ``TransformerDecoder`` with a ``DecoderSelfAttention``
    holding the SAME parameter tensors (state_dict keys and values unchanged), and set every layer's
    ``DecoderSelfAttention.precision`` (already swapped layers included) to ``precision``.  A decoder built with
    ``cross_self_attention`` (its self-attention also attends over the encoder output) raises.  Returns the
    number of layers swapped."""
    if precision not in PRECISIONS:
        raise ValueError("fbkst_b200: precision must be one of %s, got %r" % (PRECISIONS, precision))
    layers = list(getattr(decoder, "layers", []))
    if getattr(decoder, "cross_self_attention", False) or any(getattr(l, "cross_self_attention", False)
                                                               for l in layers):
        raise NotImplementedError("fbkst_b200.swap_self_attention: decoders built with cross_self_attention "
                                  "are not supported")
    swaps = []
    for layer in layers:  # build every replacement first: an unsupported layer leaves the decoder unchanged
        old = getattr(layer, "self_attn", None)
        if old is None or isinstance(old, DecoderSelfAttention):
            continue
        new = DecoderSelfAttention(old.embed_dim, old.num_heads, dropout=old.dropout,
                                   add_bias_kv=getattr(old, "bias_k", None) is not None,
                                   add_zero_attn=getattr(old, "add_zero_attn", False),
                                   self_attention=getattr(old, "self_attention", True),
                                   encoder_decoder_attention=getattr(old, "encoder_decoder_attention", False))
        for nm in ("k_proj", "v_proj", "q_proj", "out_proj"):
            getattr(new, nm).weight = getattr(old, nm).weight
            getattr(new, nm).bias = getattr(old, nm).bias
        swaps.append((layer, new))
    for layer, new in swaps:
        layer.self_attn = new
    for layer in layers:
        if isinstance(getattr(layer, "self_attn", None), DecoderSelfAttention):
            layer.self_attn.precision = precision
    return len(swaps)
