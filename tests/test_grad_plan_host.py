"""The training backward's plan (no GPU): from autograd's requests, which gradients are computed and how far down
the encoder the backward walks."""
from fbkst_b200 import train as T
from fbkst_b200.config import build_encoder
from oracle import encoder_oracle as O  # (state dicts only)

CFG = dict(embed_dim=128, ffn_dim=256, heads=2, layers=3, conv_channels=64, feat_dim=40, vocab=64,
           distance_penalty="log", ctc_layer=2, ctc_strategy="avg")


def _plan(frozen, need_x, cfg=CFG):
    enc = build_encoder(cfg, O.init_state_dict(cfg, seed=0), device="cpu")
    names = {id(p): n for n, p in enc.named_parameters()}
    ps = T.flat_parameters(enc)
    assert len(ps) == len(names)
    return T._grad_plan(enc, [not frozen(names[id(p)]) for p in ps], need_x)


def _depths(plan):
    return [d["depth"] for d in plan["layers"]]


def test_everything_requested_runs_everything():
    for need_x in (False, True):
        p = _plan(lambda n: False, need_x)
        assert _depths(p) == [6, 6, 6]
        f = p["front"]
        assert f["any"] and f["below_fc3"] and f["below_conv2"] and f["x"] == need_x
        assert all(f[k] for k in T._FRONT) and all(p["top"].values())


def test_input_gradient_alone_descends_to_conv1_and_computes_no_weight_gradient():
    p = _plan(lambda n: True, True)
    assert _depths(p) == [6, 6, 6]
    f = p["front"]
    assert f["x"] and f["below_conv2"] and not any(f[k] for k in T._FRONT)
    assert not any(v for d in p["layers"] for k, v in d.items() if k not in ("depth", "ctc"))
    assert not any(p["top"].values())


def test_frozen_bottom_stops_the_walk():
    # front end and layer 0 frozen: layer 1 runs to its first LayerNorm, layer 0 and the front end not at all
    p = _plan(lambda n: n.startswith(("convolutions.", "bn.", "fc3.", "layers.0.")), False)
    assert _depths(p) == [-1, 5, 6] and not p["front"]["any"]
    # only fc2 of layer 1 (and nothing above it but what leads there)
    p = _plan(lambda n: not n.startswith("layers.1.fc2."), False)
    assert _depths(p) == [-1, 0, 6]


def test_ctc_projection_alone_reaches_the_ctc_layer_top():
    p = _plan(lambda n: not n.startswith("ctc_fc."), False)
    assert _depths(p) == [-1, -1, 6]
    assert [d["ctc"] for d in p["layers"]] == [False, True, False]
    assert p["top"]["wc"] and p["top"]["bc"] and not p["top"]["gf"]


def test_front_end_stages():
    p = _plan(lambda n: not n.startswith("fc3."), False)
    f = p["front"]
    assert f["any"] and not f["below_fc3"] and not f["below_conv2"]
    p = _plan(lambda n: not n.startswith("bn.1."), False)
    f = p["front"]
    assert f["below_fc3"] and not f["below_conv2"] and not f["cw2"] and f["bn1_w"]


def test_separate_qkv_projections_share_one_flag():
    cfg = dict(CFG, distance_penalty=None, ctc_layer=0)
    p = _plan(lambda n: not n.startswith("layers.2.self_attn.k_proj.weight"), False, cfg)
    d = p["layers"][2]
    assert d["wqkv"] and not d["bqkv"] and not d["w2"] and d["depth"] == 4
