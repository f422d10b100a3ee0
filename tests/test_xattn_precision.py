"""CPU checks of the ``precision`` switch of the decoder cross-attention (no GPU needed): the module property,
``swap_cross_attention(..., precision=)`` and the plugin's ``--b200-cross-attention-precision`` flag."""
import argparse
import os

import pytest
import torch

from fbkst_b200.cross_attention import CrossAttention, swap_cross_attention
from oracle import ref_loader as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLUGIN = os.path.join(ROOT, "fbk-fairseq-st_b200", "fbkst_b200", "plugin")


def test_default_is_bf16_and_fp32_can_be_selected():
    m = CrossAttention(128, 2)
    assert m.precision == "bf16"
    m.precision = "fp32"
    assert m.precision == "fp32"


@pytest.mark.parametrize("bad", ["fp16", "FP32", "tf32", None, 32])
def test_unknown_precision_raises(bad):
    m = CrossAttention(128, 2)
    with pytest.raises(ValueError, match="precision"):
        m.precision = bad
    assert m.precision == "bf16"


def _decoder(n_layers, D=128, H=2):
    """What swap_cross_attention reads of a fairseq decoder: layers[i].encoder_attn with the reference
    block's attributes and projections."""
    def block():
        m = torch.nn.Module()
        m.embed_dim, m.num_heads, m.kdim, m.vdim, m.dropout = D, H, D, D, 0.0
        for nm in ("k_proj", "v_proj", "q_proj", "out_proj"):
            setattr(m, nm, torch.nn.Linear(D, D))
        return m

    dec = torch.nn.Module()
    dec.layers = torch.nn.ModuleList()
    for _ in range(n_layers):
        layer = torch.nn.Module()
        layer.encoder_attn = block()
        dec.layers.append(layer)
    return dec


def test_swap_sets_the_precision_of_every_layer():
    dec = _decoder(3)
    assert swap_cross_attention(dec, precision="fp32") == 3
    assert [type(l.encoder_attn) for l in dec.layers] == [CrossAttention] * 3
    assert [l.encoder_attn.precision for l in dec.layers] == ["fp32"] * 3
    assert swap_cross_attention(dec) == 0  # already swapped: the precision is still (re)set
    assert [l.encoder_attn.precision for l in dec.layers] == ["bf16"] * 3
    dec2 = _decoder(2)
    assert swap_cross_attention(dec2) == 2
    assert [l.encoder_attn.precision for l in dec2.layers] == ["bf16"] * 2


def test_swap_rejects_an_unknown_precision_before_swapping():
    dec = _decoder(2)
    with pytest.raises(ValueError, match="precision"):
        swap_cross_attention(dec, precision="fp16")
    assert not any(isinstance(l.encoder_attn, CrossAttention) for l in dec.layers)


@pytest.mark.skipif(not R.available(), reason="fairseq / the live reference is not importable")
def test_plugin_flag():
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

    args, model = build("--b200-cross-attention", "--b200-cross-attention-precision", "fp32")
    assert args.b200_cross_attention_precision == "fp32"
    assert [l.encoder_attn.precision for l in model.decoder.layers] == ["fp32", "fp32"]
    assert model.encoder.precision == "bf16"  # --b200-precision keeps its encoder-only meaning
    args, model = build("--b200-cross-attention")
    assert args.b200_cross_attention_precision == "bf16"
    assert [l.encoder_attn.precision for l in model.decoder.layers] == ["bf16", "bf16"]
    with pytest.raises(ValueError, match="--b200-cross-attention"):
        build("--b200-cross-attention-precision", "fp32")
