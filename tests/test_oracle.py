"""Pin the CPU oracle: golden vectors made from the live reference, the SURVEY 3.5
known-answer vector, and (when /root/reference is mounted) the live reference."""
import os

import pytest
import torch

from oracle import encoder_oracle as O
from oracle.golden import load as load_golden
from oracle import ref_loader as R


def load(golden_dir, name):
    return load_golden(os.path.join(golden_dir, name))


def assert_close(a, b, tol=1e-5):
    assert a.shape == b.shape, (a.shape, b.shape)
    err = (a.double() - b.double()).abs().max().item()
    ref = b.double().abs().max().item()
    assert err <= tol * max(ref, 1.0), (err, ref)


def test_ctc_kat_handderived():
    """SURVEY 3.5 KAT: segments, lengths and the W columns are hand-derivable."""
    lab = torch.tensor([[2, 2, 1, 1, 1, 3], [0, 0, 0, 2, 1, 1]]).t()
    mar = torch.tensor([[1, 2, .5, 1.5, 3, 1], [2, 1, .5, 4, 9, 9]]).t()
    logits = torch.zeros(6, 2, 4).scatter_(2, lab.unsqueeze(-1), mar.unsqueeze(-1))
    lengths = torch.tensor([6, 4])
    segs = O.ctc_segments(logits, lengths)
    assert segs == [[(2, 2), (1, 3), (3, 1)], [(0, 3), (2, 1)]]
    prob = torch.softmax(logits, -1).transpose(0, 1)
    W = O.ctc_weights(prob, segs, "avg", torch.float32)
    assert W.shape == (2, 6, 3)
    assert torch.allclose(W[0, :2, 0], torch.tensor([.5, .5]))
    assert torch.allclose(W[0, 2:5, 1], torch.full((3,), 1 / 3))
    assert W[0, 5, 2] == 1 and W[1, 3, 1] == 1 and W[1, 4:].abs().sum() == 0
    W = O.ctc_weights(prob, segs, "weighted", torch.float32)
    assert torch.allclose(W[0, :2, 0], torch.tensor([0.400612, 0.599388]), atol=1e-5)
    assert torch.allclose(W[0, 2:5, 1], torch.tensor([0.194470, 0.328459, 0.477071]), atol=1e-5)
    assert torch.allclose(W[1, :3, 0], torch.tensor([0.461462, 0.308427, 0.230111]), atol=1e-5)
    W = O.ctc_weights(prob, segs, "softmax", torch.float32)
    assert torch.allclose(W[0, :2, 0], torch.tensor([0.441305, 0.558695]), atol=1e-5)
    assert torch.allclose(W[0, 2:5, 1], torch.tensor([0.253095, 0.323152, 0.423753]), atol=1e-5)
    assert torch.allclose(W[1, :3, 0], torch.tensor([0.401613, 0.317229, 0.281158]), atol=1e-5)


def test_ctc_compress_golden(golden_dir):
    for c in load(golden_dir, "ctc_compress.pt"):
        out, nl, _ = O.ctc_compress(c["x"], c["logits"], c["lengths"], c["strategy"])
        assert torch.equal(nl, c["new_lengths"]), c["name"]
        assert_close(out, c["out"], 1e-6)


def test_cmvn_golden(golden_dir):
    for c in load(golden_dir, "cmvn.pt"):
        assert_close(O.cmvn(c["x"]), c["y"], 1e-6)


@pytest.mark.parametrize("name", ["enc_tiny_log.pt", "enc_tiny_nopen.pt"])
def test_encoder_golden(golden_dir, name):
    fx = load(golden_dir, name)
    cfg = fx["cfg"]
    hook = O.bump_hook(fx["bump_labels"], fx["bump_margin"]) if "bump_labels" in fx else None
    for s, ref in fx["outputs"].items():
        out = O.encoder_forward(fx["state_dict"], dict(cfg, ctc_strategy=s), fx["src_tokens"],
                                fx["src_lengths"], return_all_hiddens=True, ctc_logits_hook=hook)
        assert_close(out["encoder_out"], ref["encoder_out"], 1e-5)
        assert torch.equal(out["src_lengths"], ref["src_lengths"])
        if ref["encoder_padding_mask"] is None:
            assert out["encoder_padding_mask"] is None
        else:
            assert torch.equal(out["encoder_padding_mask"], ref["encoder_padding_mask"])
        assert len(out["encoder_states"]) == len(ref["encoder_states"])
        for a, b in zip(out["encoder_states"], ref["encoder_states"]):
            assert_close(a, b, 1e-5)
        if cfg.get("ctc_layer", 0) > 0:
            assert_close(out["ctc_out"], ref["ctc_out"], 1e-5)
            assert torch.equal(out["ctc_padding_mask"], ref["ctc_padding_mask"])


@pytest.mark.reference
@pytest.mark.skipif(not R.available(), reason="live reference not mounted")
def test_oracle_vs_live_reference_cfg1_shape():
    """BASELINE cfg1 model (6L d256 h4 ffn768, avg@4, no penalty) at a reduced batch,
    oracle vs the live reference module."""
    cfg = dict(embed_dim=256, ffn_dim=768, heads=4, layers=6, conv_channels=64, feat_dim=40,
               vocab=105, distance_penalty=None, ctc_layer=4, ctc_strategy="avg")
    enc = R.build_reference_encoder(cfg, seed=3)
    x, lens = O.synthetic_batch([200, 190, 97, 50], 40, seed=99)
    labels = O.synthetic_ctc_bump(50, 4, 105, seed=1)
    hook = O.bump_hook(labels, 25.0)
    h = enc.ctc_fc.register_forward_hook(lambda m, i, o: hook(o))
    ref = R.run_reference_encoder(enc, x, lens)
    h.remove()
    out = O.encoder_forward(enc.state_dict(), cfg, x, lens, ctc_logits_hook=hook)
    assert torch.equal(out["src_lengths"], ref.src_lengths)
    assert_close(out["encoder_out"], ref.encoder_out, 1e-5)
    assert torch.equal(out["encoder_padding_mask"], ref.encoder_padding_mask)


def test_init_state_dict_matches_reference_keys(golden_dir):
    """Keys and shapes of the reference encoder's state_dict for this configuration, as stored by
    oracle/make_golden.py in enc_tiny_log.pt."""
    cfg = dict(embed_dim=128, ffn_dim=128, heads=2, layers=2, conv_channels=64, feat_dim=40,
               vocab=48, distance_penalty="log", ctc_layer=1, ctc_strategy="avg")
    fx = load(golden_dir, "enc_tiny_log.pt")
    assert {k: v for k, v in fx["cfg"].items() if k != "dropout"} == cfg
    ref = fx["state_dict"]
    sd = O.init_state_dict(cfg)
    assert set(sd.keys()) == set(ref.keys())
    for k in ref:
        assert tuple(sd[k].shape) == tuple(ref[k].shape), k


# ------------------------------------------------------------------ next row N2: collater
def _kat_samples():
    """tests/speech_recognition/test_collaters.py:23-31 of the reference."""
    import numpy as np
    frames1 = np.array([[7, 8], [9, 10]])
    frames2 = np.array([[1, 2], [3, 4], [5, 6]])
    target1 = np.array([4, 2, 3, 1])
    target2 = np.array([3, 2, 1])
    return [{"id": 0, "data": [frames1, target1]}, {"id": 1, "data": [frames2, target2]}]


def test_collate_oracle_reference_kat():
    """The reference's own known-answer vector (test_collaters.py:33-50) pins the collate oracle."""
    from oracle import collate_oracle as C
    batch = C.collate(_kat_samples(), pad_index=0, eos_index=1, move_eos_to_beginning=True)
    assert batch["id"].tolist() == [1, 0]
    assert batch["ntokens"] == 7 and batch["nsentences"] == 2
    assert batch["net_input"]["src_tokens"].tolist() == [[[1, 2], [3, 4], [5, 6]], [[7, 8], [9, 10], [0, 0]]]
    assert batch["net_input"]["prev_output_tokens"].tolist() == [[1, 3, 2, 0], [1, 4, 2, 3]]
    assert batch["net_input"]["src_lengths"].tolist() == [3, 2]
    assert batch["target"].tolist() == [[3, 2, 1, 0], [4, 2, 3, 1]]


@pytest.mark.skipif(not R.available(), reason="live reference not mounted")
def test_collate_oracle_vs_live_reference():
    from oracle import collate_oracle as C
    R.load()
    from examples.speech_recognition.data.collaters import Seq2SeqCollater
    g = torch.Generator().manual_seed(3)
    samples = []
    for i, n in enumerate([17, 40, 40, 5, 23]):
        tl = 3 + i
        samples.append({"id": i, "data": [torch.randn(n, 8, generator=g).numpy(),
                                          torch.randint(3, 50, (tl,), generator=g).numpy()]})
    ref = Seq2SeqCollater(0, 1, pad_index=1, eos_index=2).collate(samples)
    got = C.collate(samples, pad_index=1, eos_index=2, move_eos_to_beginning=True)
    assert torch.equal(ref["net_input"]["src_lengths"], got["net_input"]["src_lengths"])
    # ties (two utterances of 40 frames) may be ordered either way by torch.sort: compare as sets
    assert sorted(ref["id"].tolist()) == sorted(got["id"].tolist())
    for k in range(5):
        j = got["id"].tolist().index(int(ref["id"][k]))
        assert torch.equal(ref["net_input"]["src_tokens"][k], got["net_input"]["src_tokens"][j])
        assert torch.equal(ref["net_input"]["prev_output_tokens"][k], got["net_input"]["prev_output_tokens"][j])
        assert torch.equal(ref["target"][k], got["target"][j])


@pytest.mark.reference
@pytest.mark.skipif(not R.available(), reason="live reference not mounted")
@pytest.mark.parametrize("penalty,strategy", [("log", "weighted"), (None, "avg")])
def test_oracle_gradients_vs_live_reference(penalty, strategy):
    """Gradient pin (scope row T): torch.autograd through the oracle equals torch.autograd through the LIVE
    reference module in eval() + grad mode (BatchNorm running statistics, no dropout: the deterministic
    setting), for every parameter -- so the GPU gradient-parity tests (tests/test_gpu_train.py), which
    compare with the oracle, are anchored to the reference itself."""
    import warnings
    cfg = dict(embed_dim=128, ffn_dim=256, heads=2, layers=3, conv_channels=64, feat_dim=40, vocab=64,
               distance_penalty=penalty, ctc_layer=2, ctc_strategy=strategy)
    enc = R.build_reference_encoder(cfg, seed=3)
    sd = {k: v.detach().clone() for k, v in enc.state_dict().items()}
    x, lens = O.synthetic_batch([97, 64, 30], 40, seed=11)
    labels = O.synthetic_ctc_bump(25, 3, 64, seed=2)
    hook = O.bump_hook(labels, 30.0)
    enc.ctc_fc.register_forward_hook(lambda m, i, o: hook(o))
    g = torch.Generator().manual_seed(0)
    with R.cpu_cuda_noop(), R.grad_shims(), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = enc(x, lens, return_all_hiddens=True)
        r_out = torch.randn(out.encoder_out.shape, generator=g)
        r_ctc = torch.randn(out.ctc_out.shape, generator=g) * 0.05
        ((out.encoder_out * r_out).sum() + (out.ctc_out * r_ctc).sum()).backward()
    leaf = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k
                and "_float_tensor" not in k else v) for k, v in sd.items()}
    ref = O.encoder_forward(leaf, cfg, x, lens, ctc_logits_hook=hook)
    assert_close(ref["encoder_out"].detach(), out.encoder_out.detach(), 1e-5)
    ((ref["encoder_out"] * r_out).sum() + (ref["ctc_out"] * r_ctc).sum()).backward()
    n = 0
    for name, p in enc.named_parameters():
        assert p.grad is not None and leaf[name].grad is not None, name
        assert_close(leaf[name].grad, p.grad, 2e-4)
        n += 1
    assert n >= 40
