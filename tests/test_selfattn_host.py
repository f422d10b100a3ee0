"""Host logic of the N5 row (no GPU): constructor errors, the precision switch, swap_self_attention and the plugin
flags of DecoderSelfAttention, the ancestry-table form of reorder_incremental_state, no CPU fallback."""
import argparse
import os

import pytest
import torch

from fbkst_b200.self_attention import DecoderSelfAttention, swap_self_attention
from oracle import ref_loader as R
from oracle import self_attention_oracle as SA

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLUGIN = os.path.join(ROOT, "fbk-fairseq-st_b200", "fbkst_b200", "plugin")


@pytest.mark.parametrize("kwargs", [
    dict(self_attention=False), dict(encoder_decoder_attention=True), dict(add_bias_kv=True),
    dict(add_zero_attn=True), dict(q_noise=0.1), dict(bias=False), dict(kdim=64), dict(vdim=64)])
def test_unsupported_settings_raise(kwargs):
    with pytest.raises(NotImplementedError):
        DecoderSelfAttention(128, 2, **kwargs)


@pytest.mark.parametrize("D,H", [(96, 2), (128, 4), (17 * 64, 17)])  # head_dim 48, head_dim 32, 17 heads
def test_head_shape_limits_raise(D, H):
    with pytest.raises(NotImplementedError):
        DecoderSelfAttention(D, H)


def test_reference_constructor_and_state_dict():
    """MultiheadAttention(embed_dim, heads, dropout=..., self_attention=True): same keys and shapes, strict load."""
    m = DecoderSelfAttention(256, 4, dropout=0.1, self_attention=True)
    P = SA.init_params(256, 0)
    assert {k: tuple(v.shape) for k, v in P.items()} == {k: tuple(v.shape) for k, v in m.state_dict().items()}
    m.load_state_dict(P, strict=True)
    assert m.dropout == 0.1 and m.self_attention and not m.encoder_decoder_attention
    assert list(m.state_dict().keys())[:2] == ["k_proj.weight", "k_proj.bias"]  # registration order


def test_default_is_bf16_and_fp32_can_be_selected():
    m = DecoderSelfAttention(128, 2)
    assert m.precision == "bf16"
    m.precision = "fp32"
    assert m.precision == "fp32"


@pytest.mark.parametrize("bad", ["fp16", "FP32", "tf32", None, 32])
def test_unknown_precision_raises(bad):
    m = DecoderSelfAttention(128, 2)
    with pytest.raises(ValueError, match="precision"):
        m.precision = bad
    assert m.precision == "bf16"


def test_no_cpu_fallback_and_no_backward():
    m = DecoderSelfAttention(128, 2).eval()
    q = torch.randn(1, 2, 128)
    with pytest.raises(RuntimeError):
        m(q, q, q, incremental_state={})
    m.train()
    with pytest.raises(NotImplementedError):
        m(q, q, q)


def test_reorder_moves_only_the_ancestry_table():
    m = DecoderSelfAttention(128, 2)
    inc = {}
    cache = torch.randn(4, 6, 3 * 128)
    pad = torch.zeros(4, 6, dtype=torch.uint8)
    anc = torch.arange(6, dtype=torch.int32).repeat(4, 1)
    m._set_input_buffer(inc, dict(fbkst_cache=cache, fbkst_anc=anc, fbkst_pad=pad, fbkst_steps=3))
    want = anc.clone()
    for order in ([1, 0, 3, 2, 5, 4], [5, 4, 3, 2, 1, 0], [0, 1, 4, 5], [3, 2], [0]):
        order = torch.tensor(order)
        assert m.reorder_incremental_state(inc, order) is inc
        want = want[:, order]
        buf = m._get_input_buffer(inc)
        assert torch.equal(buf["fbkst_anc"], want)
        assert buf["fbkst_cache"] is cache and buf["fbkst_pad"] is pad and buf["fbkst_steps"] == 3


def _decoder(n_layers, D=128, H=2, cross_self_attention=False):
    """What swap_self_attention reads of a fairseq decoder: layers[i].self_attn with the reference block's
    attributes and projections, in the reference's registration order."""
    def block():
        m = torch.nn.Module()
        m.embed_dim, m.num_heads, m.dropout = D, H, 0.1
        m.bias_k, m.add_zero_attn = None, False
        m.self_attention, m.encoder_decoder_attention = not cross_self_attention, False
        for nm in ("k_proj", "v_proj", "q_proj", "out_proj"):
            setattr(m, nm, torch.nn.Linear(D, D))
        return m

    dec = torch.nn.Module()
    dec.cross_self_attention = cross_self_attention
    dec.layers = torch.nn.ModuleList()
    for _ in range(n_layers):
        layer = torch.nn.Module()
        layer.self_attn = block()
        dec.layers.append(layer)
    return dec


def test_swap_keeps_state_dict_and_is_idempotent():
    dec = _decoder(3)
    before = {k: v.clone() for k, v in dec.state_dict().items()}
    params = [l.self_attn.q_proj.weight for l in dec.layers]
    assert swap_self_attention(dec) == 3
    assert [type(l.self_attn) for l in dec.layers] == [DecoderSelfAttention] * 3
    after = dec.state_dict()
    assert list(after.keys()) == list(before.keys())
    assert all(torch.equal(after[k], before[k]) for k in before)
    assert all(l.self_attn.q_proj.weight is p for l, p in zip(dec.layers, params))
    assert [l.self_attn.dropout for l in dec.layers] == [0.1] * 3
    swapped = [l.self_attn for l in dec.layers]
    assert swap_self_attention(dec, precision="fp32") == 0  # already swapped: only the precision is set
    assert [l.self_attn for l in dec.layers] == swapped
    assert [l.self_attn.precision for l in dec.layers] == ["fp32"] * 3
    assert swap_self_attention(dec) == 0
    assert [l.self_attn.precision for l in dec.layers] == ["bf16"] * 3


def test_swap_rejects_before_swapping():
    dec = _decoder(2)
    with pytest.raises(ValueError, match="precision"):
        swap_self_attention(dec, precision="fp16")
    assert not any(isinstance(l.self_attn, DecoderSelfAttention) for l in dec.layers)
    dec = _decoder(2, cross_self_attention=True)
    with pytest.raises(NotImplementedError, match="cross_self_attention"):
        swap_self_attention(dec)
    assert not any(isinstance(l.self_attn, DecoderSelfAttention) for l in dec.layers)
    dec = _decoder(2)
    dec.layers[1].self_attn.bias_k = torch.nn.Parameter(torch.zeros(1, 1, 128))  # add_bias_kv in one layer
    with pytest.raises(NotImplementedError):
        swap_self_attention(dec)
    assert not any(isinstance(l.self_attn, DecoderSelfAttention) for l in dec.layers)


@pytest.mark.skipif(not R.available(), reason="fairseq / the live reference is not importable")
def test_plugin_flags():
    R.load()
    from fairseq import options, utils
    from fairseq.models import MODEL_REGISTRY
    utils.import_user_module(argparse.Namespace(user_dir=PLUGIN))

    def build(*extra):
        parser = options.get_training_parser()
        args = options.parse_args_and_arch(parser, [
            "/tmp/nodata", "--user-dir", PLUGIN, "--arch", "conv_transformer_b200",
            "--task", "speech_translation_with_transcription", "--criterion", "ctc_multi_loss",
            "--underlying-criterion", "label_smoothed_cross_entropy", "--ctc-encoder-layer", "1",
            "--ctc-compress-out", "--ctc-compress-strategy", "avg", "--no-attn-2d",
            "--distance-penalty", "log", "--input-feat-per-channel", "40", "--encoder-layers", "2",
            "--decoder-layers", "2", "--max-tokens", "1000", "--skip-normalization"] + list(extra))
        task = argparse.Namespace(source_dictionary=R.make_dictionary(60), target_dictionary=R.make_dictionary(70))
        return args, MODEL_REGISTRY["conv_transformer_b200"].build_model(args, task)

    args, model = build("--b200-self-attention", "--b200-self-attention-precision", "fp32")
    assert [l.self_attn.precision for l in model.decoder.layers] == ["fp32", "fp32"]
    assert model.encoder.precision == "bf16"
    assert not any(type(l.encoder_attn).__name__ == "CrossAttention" for l in model.decoder.layers)
    args, model = build("--b200-self-attention")
    assert args.b200_self_attention_precision == "bf16"
    assert [type(l.self_attn) for l in model.decoder.layers] == [DecoderSelfAttention] * 2
    args, model = build()
    assert not any(isinstance(l.self_attn, DecoderSelfAttention) for l in model.decoder.layers)
    with pytest.raises(ValueError, match="--b200-self-attention"):
        build("--b200-self-attention-precision", "fp32")
