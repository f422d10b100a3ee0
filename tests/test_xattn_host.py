"""Host logic of the N4 row (no GPU): beam tags left by reorder_encoder_out, the row-map form of
reorder_incremental_state, state_dict compatibility with the reference block, no CPU fallback."""
import os

import pytest
import torch

from fbkst_b200.cross_attention import CrossAttention, beam_source, reorder_tagged, swap_cross_attention
from fbkst_b200.encoder import ConvolutionalTransformerEncoder, EncoderOut
from oracle import cross_attention_oracle as X
from oracle.golden import load as load_golden


def _enc_out(S=7, U=3, D=8):
    g = torch.Generator().manual_seed(0)
    x = torch.randn(S, U, D, generator=g)
    m = torch.zeros(U, S, dtype=torch.bool)
    m[1, 4:] = True
    return EncoderOut(x, m, None, None, None, None)


@pytest.mark.parametrize("lazy", [False, True])
def test_reorder_encoder_out_values_and_tags(lazy):
    """Eager: bit-identical to the reference gather (conv_transformer.py:329-338) through a chain of
    reorders; both modes: the tag always points at the ORIGINAL tensors with composed rows."""
    eo = _enc_out()
    enc = ConvolutionalTransformerEncoder.__new__(ConvolutionalTransformerEncoder)  # method needs no state
    torch.nn.Module.__init__(enc)
    enc.lazy_beam_reorder = lazy
    o1 = torch.tensor([0, 0, 1, 1, 2, 2])
    o2 = torch.tensor([1, 0, 4, 5])
    r1 = enc.reorder_encoder_out(eo, o1)
    r2 = enc.reorder_encoder_out(r1, o2)
    want_x, want_m = X.reorder_encoder_out(*X.reorder_encoder_out(eo.encoder_out, eo.encoder_padding_mask, o1), o2)
    base, rows = beam_source(r2.encoder_out)
    mbase, mrows = beam_source(r2.encoder_padding_mask)
    assert base is eo.encoder_out or base.data_ptr() == eo.encoder_out.data_ptr()
    assert rows.tolist() == o1[o2].tolist() and rows is mrows
    assert mbase.data_ptr() == eo.encoder_padding_mask.data_ptr()
    if lazy:
        assert r2.encoder_out.shape == eo.encoder_out.shape  # nothing was replicated
    else:
        assert torch.equal(r2.encoder_out, want_x) and torch.equal(r2.encoder_padding_mask, want_m)
    # the first result is untouched by the second reorder
    assert beam_source(r1.encoder_out)[1].tolist() == o1.tolist()


def test_row_map_reorder_follows_the_reference_rule():
    """multihead_attention.py:416: same-size new_order leaves the cache alone; a shrinking batch
    gathers.  Checked against the oracle's restatement acting on a per-row cache."""
    m = CrossAttention(128, 2)
    inc = {}
    row_map = torch.tensor([0, 0, 1, 1, 2, 2], dtype=torch.int32)
    m._set_input_buffer(inc, dict(fbkst_kv=None, fbkst_mask=None, fbkst_row_map=row_map))
    ref = {"prev_key": row_map.clone().view(6, 1, 1, 1).float()}
    for order in ([1, 0, 3, 2, 5, 4], [5, 4, 3, 2, 1, 0], [0, 1, 4, 5], [3, 2], [0]):
        order = torch.tensor(order)
        m.reorder_incremental_state(inc, order)
        X.reorder_state(ref, order)
        assert m._get_input_buffer(inc)["fbkst_row_map"].tolist() == ref["prev_key"].flatten().int().tolist()


def test_no_cpu_fallback_and_no_backward():
    m = CrossAttention(128, 2).eval()
    q, k = torch.randn(1, 2, 128), torch.randn(5, 2, 128)
    with pytest.raises(RuntimeError):
        m(q, k, k, static_kv=True)
    m.train()
    with pytest.raises(NotImplementedError):
        m(q, k, k, static_kv=True)
    with pytest.raises(NotImplementedError):
        CrossAttention(96, 2)  # head_dim 48


def test_state_dict_is_the_reference_blocks(golden_dir):
    """Parameters of the reference's MultiheadAttention(256, 4, kdim=192, vdim=192,
    encoder_decoder_attention=True), as oracle/make_golden_xattn.py loaded them into it with strict=True
    (xattn.pt, case nomask_heads): same keys and shapes here, strict load, and swap_cross_attention
    keeps a decoder's state_dict keys and parameter tensors."""
    case = load_golden(os.path.join(golden_dir, "xattn.pt"))["nomask_heads"]
    D, H, kdim, params = case["D"], case["H"], case["kdim"], case["params"]
    ours = CrossAttention(D, H, kdim=kdim, vdim=kdim)
    assert {k: tuple(v.shape) for k, v in params.items()} == \
           {k: tuple(v.shape) for k, v in ours.state_dict().items()}
    ours.load_state_dict(params, strict=True)

    ref = torch.nn.Module()  # what swap_cross_attention reads of a MultiheadAttention, in its layout
    ref.embed_dim, ref.num_heads, ref.kdim, ref.vdim, ref.dropout = D, H, kdim, kdim, 0.0
    for nm in ("k_proj", "v_proj", "q_proj", "out_proj"):  # multihead_attention.py registration order
        w = params[nm + ".weight"]
        setattr(ref, nm, torch.nn.Linear(w.shape[1], w.shape[0]))
    ref.load_state_dict(params, strict=True)

    class _Layer(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.encoder_attn = ref

    class _Dec(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.layers = torch.nn.ModuleList([_Layer()])

    dec = _Dec()
    keys = list(dec.state_dict().keys())
    assert swap_cross_attention(dec) == 1
    assert isinstance(dec.layers[0].encoder_attn, CrossAttention)
    assert list(dec.state_dict().keys()) == keys
    assert dec.layers[0].encoder_attn.k_proj.weight is ref.k_proj.weight
