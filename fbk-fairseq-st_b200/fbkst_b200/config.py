"""Build the encoder from a plain config dict (tests, bench, smoke) without fairseq's parser.

The Namespace carries exactly the fields the reference ctor reads
(examples/speech_recognition/models/conv_transformer.py:134-193) with the defaults of
``base_architecture`` (:429-466) for the flags this path supports."""
import argparse


class DictStub:
    """len()-only stand-in for fairseq's Dictionary (the encoder reads only ``len(dictionary)``)."""

    def __init__(self, n):
        self.n = n

    def __len__(self):
        return self.n


def make_args(cfg):
    a = argparse.Namespace()
    a.encoder_embed_dim = cfg["embed_dim"]
    a.encoder_ffn_embed_dim = cfg["ffn_dim"]
    a.encoder_attention_heads = cfg["heads"]
    a.encoder_layers = cfg["layers"]
    a.encoder_convolutions = "[(%d, 3, 3)] * 2" % cfg.get("conv_channels", 64)
    a.input_feat_per_channel = cfg["feat_dim"]
    a.distance_penalty = "log" if cfg.get("distance_penalty", "log") == "log" else False
    a.attn_2d = False
    a.ctc_compress_out = cfg.get("ctc_layer", 0) > 0
    a.ctc_compress_strategy = cfg.get("ctc_strategy", "avg")
    a.ctc_encoder_layer = cfg.get("ctc_layer", 0)
    a.criterion = "ctc_multi_loss"
    a.max_source_positions = cfg.get("max_source_positions", 100000)
    a.encoder_layerdrop = 0.0
    a.dropout = cfg.get("dropout", 0.1)
    a.attention_dropout = cfg.get("attention_dropout", 0.1)  # base_architecture defaults (:432-433)
    a.relu_dropout = cfg.get("relu_dropout", 0.1)
    a.encoder_normalize_before = True
    a.encoder_learned_pos = bool(cfg.get("learned_pos", False))
    a.no_token_positional_embeddings = False
    a.layernorm_embedding = False
    return a


def build_encoder(cfg, state_dict=None, device="cuda:0"):
    from .encoder import ConvolutionalTransformerEncoder
    enc = ConvolutionalTransformerEncoder(make_args(cfg), DictStub(cfg["vocab"]),
                                          audio_features=cfg["feat_dim"])
    if state_dict is not None:
        enc.load_state_dict(state_dict, strict=True)
    # An inference encoder: eval() and frozen parameters.  (As with any nn.Module, a forward with gradients
    # enabled and parameters that require them builds the differentiable chain -- fbkst_b200.train -- so
    # callers that want gradients re-enable requires_grad; fairseq's generate / validate run under no_grad.)
    for p in enc.parameters():
        p.requires_grad_(False)
    enc.precision = cfg.get("precision", "bf16")  # "fp32": split-TF32 inference path (encoder.precision)
    return enc.to(device).eval()
