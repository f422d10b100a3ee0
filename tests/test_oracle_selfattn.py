"""Pins oracle/self_attention_oracle.py (CPU, fp64): the step-by-step torch.cat restatement equals PyTorch's own
multi-head attention over the whole sequence under a causal mask, and through random beam reorders and a
shrinking batch every hypothesis's output equals a causal recomputation over its own token history rebuilt from
the back-pointers.  Where fairseq is importable, the oracle is also compared with the live MultiheadAttention."""
import pytest
import torch
import torch.nn.functional as F

from oracle import ref_loader as R
from oracle import self_attention_oracle as SA

D, H = 128, 2


def _params(seed):
    return {k: v.double() for k, v in SA.init_params(D, seed).items()}


def _mha_causal(P, x, key_padding_mask=None):
    """torch.nn.functional.multi_head_attention_forward over the whole (T, bsz, D) sequence, causal."""
    T = x.shape[0]
    if key_padding_mask is not None:  # the same (float) mask type as attn_mask
        key_padding_mask = torch.zeros(key_padding_mask.shape, dtype=x.dtype).masked_fill(key_padding_mask,
                                                                                          float("-inf"))
    return F.multi_head_attention_forward(
        x, x, x, D, H, None, torch.cat([P["q_proj.bias"], P["k_proj.bias"], P["v_proj.bias"]]), None, None, False,
        0.0, P["out_proj.weight"], P["out_proj.bias"], training=False, key_padding_mask=key_padding_mask,
        need_weights=True, attn_mask=SA.future_mask(T, torch.float64), use_separate_proj_weight=True,
        q_proj_weight=P["q_proj.weight"], k_proj_weight=P["k_proj.weight"], v_proj_weight=P["v_proj.weight"])


def test_stepwise_equals_causal_mha_fp64():
    P = _params(1)
    g = torch.Generator().manual_seed(2)
    T, bsz = 9, 4
    x = torch.randn(T, bsz, D, generator=g, dtype=torch.float64)
    ref, ref_w = _mha_causal(P, x)
    st = {}
    for t in range(T):
        a, w = SA.self_attention(P, H, x[t:t + 1], state=st)
        assert (a[0] - ref[t]).abs().max().item() <= 1e-10
        assert (w[:, 0] - ref_w[:, t, :t + 1]).abs().max().item() <= 1e-10
    # the full call under the future mask is the same computation
    a, w = SA.self_attention(P, H, x, attn_mask=SA.future_mask(T, torch.float64))
    assert (a - ref).abs().max().item() <= 1e-10 and (w - ref_w).abs().max().item() <= 1e-10


def test_stepwise_padding_equals_causal_mha_fp64():
    """Per-step key padding appended step by step (zeros stand in for steps without a mask)."""
    P = _params(3)
    g = torch.Generator().manual_seed(4)
    T, bsz = 6, 3
    x = torch.randn(T, bsz, D, generator=g, dtype=torch.float64)
    kpm = torch.zeros(bsz, T, dtype=torch.bool)
    kpm[1, 2] = kpm[2, 4] = True
    ref, _ = _mha_causal(P, x, key_padding_mask=kpm)
    st = {}
    for t in range(T):
        m = kpm[:, t:t + 1] if t >= 2 else None  # steps 0 and 1 carry no mask
        a, _ = SA.self_attention(P, H, x[t:t + 1], key_padding_mask=m, state=st)
        assert (a[0] - ref[t]).abs().max().item() <= 1e-10


def test_reorders_and_shrinking_batch_follow_each_hypothesis_history():
    P = _params(5)
    g = torch.Generator().manual_seed(6)
    bsz, beam = 3, 4
    n = bsz * beam
    st, hist = {}, [[] for _ in range(n)]
    for t in range(10):
        if t > 0:
            if t in (4, 7):  # sentences finish: the batch shrinks
                keep = torch.randperm(n, generator=g)[: n - beam]
                order = keep.sort().values
            else:  # same-size reorder: each sentence's beam picks parents among its own hypotheses
                order = torch.arange(n).view(-1, beam)
                order = order.gather(1, torch.randint(0, beam, order.shape, generator=g)).view(-1)
            SA.reorder_state(st, order)
            hist = [list(hist[o]) for o in order.tolist()]
            n = order.numel()
        x = torch.randn(1, n, D, generator=g, dtype=torch.float64)
        for b in range(n):
            hist[b].append(x[0, b])
        a, _ = SA.self_attention(P, H, x, state=st)
        for b in range(n):
            seq = torch.stack(hist[b]).view(-1, 1, D)
            full, _ = SA.self_attention(P, H, seq, attn_mask=SA.future_mask(seq.shape[0], torch.float64))
            assert (a[0, b] - full[-1, 0]).abs().max().item() <= 1e-10, (t, b)


def test_oracle_matches_live_multihead_attention():
    if R.available():  # the reference tree carries its fairseq
        R.load()
    fairseq_mha = pytest.importorskip("fairseq.modules.multihead_attention")
    P = {k: v.float() for k, v in SA.init_params(D, 7).items()}
    m = fairseq_mha.MultiheadAttention(D, H, self_attention=True).eval()
    m.load_state_dict(P, strict=True)
    g = torch.Generator().manual_seed(8)
    n = 6
    inc, st = {}, {}
    with torch.no_grad():
        for t in range(5):
            if t > 0:
                order = torch.randint(0, n, (n if t != 3 else n - 2,), generator=g)
                m.reorder_incremental_state(inc, order)
                SA.reorder_state(st, order)
                n = order.numel()
            x = torch.randn(1, n, D, generator=g)
            want, _ = SA.self_attention(P, H, x, state=st)
            got, _ = m(x, x, x, incremental_state=inc, need_weights=False)
            assert (got - want).abs().max().item() <= 1e-5
