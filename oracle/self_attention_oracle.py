"""CPU restatement of the decoder's self-attention on its incremental path and of the beam reorder of its
cache -- TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``): imported by ``tests/``, never by the product.

No live-reference golden vectors pin this file: ``tests/test_oracle_selfattn.py`` pins it against
``torch.nn.functional.multi_head_attention_forward`` (causal, fp64) and against a full recomputation of every
hypothesis over its own token history, and against the live ``MultiheadAttention`` where fairseq is importable.

Reference lines followed (``fairseq/modules/multihead_attention.py``, ``self_attention=True``):
  :194-209   q, k, v = q_proj / k_proj / v_proj of the query; q *= head_dim**-0.5
  :229-246   (T, B, D) -> (B*H, T, hd) head split
  :248-281   incremental state: prev_key / prev_value (bsz, H, t, hd) concatenated with the new step
             (torch.cat on the time axis), prev_key_padding_mask appended (_append_prev_key_padding_mask:
             zeros stand in for a missing side)
  :317-335   scores = q k^T ; + attn_mask ; padding keys -> -inf
  :340-353   fp32 softmax ; attn = P v ; out_proj
  :355-362   weights (H, bsz, tgt, src) or their mean over heads
  :407-420   reorder_incremental_state: every cached tensor index_select(0, new_order) (the same-size skip is
             for encoder-decoder attention only)
"""
import torch
import torch.nn.functional as F

from .cross_attention_oracle import _split_heads, init_params as _init_params


def init_params(D, seed):
    """Parameters of one self-attention block (names as in the reference state_dict)."""
    return _init_params(D, D, seed)


def future_mask(T, dtype=torch.float32):
    """fairseq's buffered_future_mask: -inf strictly above the diagonal, 0 elsewhere."""
    return torch.triu(torch.full((T, T), float("-inf"), dtype=dtype), 1)


def _append_prev_key_padding_mask(kpm, prev, bsz, src_len):
    if prev is not None and kpm is not None:
        return torch.cat([prev.float(), kpm.float()], dim=1)
    if prev is not None:
        return torch.cat([prev.float(), torch.zeros(bsz, src_len - prev.size(1))], dim=1)
    if kpm is not None:
        return torch.cat([torch.zeros(bsz, src_len - kpm.size(1)), kpm.float()], dim=1)
    return None


def self_attention(P, H, query, key_padding_mask=None, state=None, attn_mask=None, need_weights=True,
                   need_head_weights=False):
    """One call of the block on ``query`` (tgt, bsz, D).  ``state`` (a dict, mutated) is the layer's
    incremental buffer: the new keys / values are appended to ``prev_key`` / ``prev_value`` with torch.cat.
    Returns (attn (tgt, bsz, D), weights or None)."""
    tgt, bsz, D = query.shape
    hd = D // H
    q = _split_heads(F.linear(query, P["q_proj.weight"], P["q_proj.bias"]) * hd ** -0.5, H)
    k = _split_heads(F.linear(query, P["k_proj.weight"], P["k_proj.bias"]), H)
    v = _split_heads(F.linear(query, P["v_proj.weight"], P["v_proj.bias"]), H)
    if state is not None:
        prev_mask = None
        if "prev_key" in state:
            k = torch.cat([state["prev_key"].view(bsz * H, -1, hd), k], dim=1)
            v = torch.cat([state["prev_value"].view(bsz * H, -1, hd), v], dim=1)
            prev_mask = state.get("prev_key_padding_mask")
        key_padding_mask = _append_prev_key_padding_mask(key_padding_mask, prev_mask, bsz, k.size(1))
        state["prev_key"] = k.view(bsz, H, -1, hd)
        state["prev_value"] = v.view(bsz, H, -1, hd)
        state["prev_key_padding_mask"] = key_padding_mask
    S = k.size(1)
    w = torch.bmm(q, k.transpose(1, 2))  # (bsz*H, tgt, S)
    if attn_mask is not None:
        w = w + attn_mask.to(w.dtype).unsqueeze(0)
    if key_padding_mask is not None:
        w = w.view(bsz, H, tgt, S).masked_fill(
            key_padding_mask.view(bsz, 1, 1, S).to(torch.bool), float("-inf")).view(bsz * H, tgt, S)
    # fp32 softmax (utils.softmax); fp64 scores stay fp64 so that fp64 pinning tests are exact to ~1e-15
    p = torch.softmax(w if w.dtype == torch.float64 else w.float(), dim=-1).type_as(w)
    a = torch.bmm(p, v).transpose(0, 1).contiguous().view(tgt, bsz, D)
    a = F.linear(a, P["out_proj.weight"], P["out_proj.bias"])
    weights = None
    if need_weights:
        weights = p.view(bsz, H, tgt, S).transpose(1, 0)
        if not need_head_weights:
            weights = weights.mean(dim=0)
    return a, weights


def reorder_state(state, new_order):
    """multihead_attention.py:407-420 for a self-attention block: every cached tensor is gathered along the
    hypothesis dimension, at every call."""
    for k in list(state.keys()):
        if state[k] is not None:
            state[k] = state[k].index_select(0, new_order)
    return state
