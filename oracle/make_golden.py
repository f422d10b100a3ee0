"""Regenerate ``tests/golden/*.pt`` from the LIVE reference -- TEST INFRASTRUCTURE ONLY.

Run in the build container (needs ``/root/reference``):

    python -m oracle.make_golden

Each fixture stores inputs, the reference's own ``state_dict`` and the outputs
of the reference's own ``ConvolutionalTransformerEncoder.forward`` (eval mode,
CPU fp32, shims of ``oracle/ref_loader.py``).  They are committed, so the tests
need no reference; ``oracle/golden.py`` stores a fixture of more than 1 MB as parts.
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle import encoder_oracle as O  # noqa: E402
from oracle import golden  # noqa: E402
from oracle import ref_loader as R  # noqa: E402

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

TINY = dict(embed_dim=128, ffn_dim=128, heads=2, layers=2, conv_channels=64, feat_dim=40,
            vocab=48, distance_penalty="log", ctc_layer=1, ctc_strategy="avg", dropout=0.1)
TINY_NOPEN = dict(TINY, distance_penalty=None, layers=1, ctc_layer=0)


def out_to_dict(out):
    d = {}
    for k in out._fields:
        v = getattr(out, k)
        if k == "src_tokens":
            continue
        d[k] = v
    return d


def encoder_fixture(cfg, lengths, seed, strategies, margin=30.0):
    enc = R.build_reference_encoder(cfg, seed=seed)
    sd = {k: v.clone() for k, v in enc.state_dict().items()}
    x, lens = O.synthetic_batch(lengths, cfg["feat_dim"], seed=1234 + seed)
    fx = dict(cfg=cfg, state_dict=sd, src_tokens=x, src_lengths=lens, outputs={})
    if cfg.get("ctc_layer", 0) > 0:
        T1 = -(-max(lengths) // 2)
        Lp = -(-T1 // 2)
        labels = O.synthetic_ctc_bump(Lp, len(lengths), cfg["vocab"], seed=7 + seed)
        fx["bump_labels"], fx["bump_margin"] = labels, margin
        hook = O.bump_hook(labels, margin)
        enc.ctc_fc.register_forward_hook(lambda m, i, o: hook(o))
    import examples.speech_recognition.models.conv_transformer as ct
    for s in strategies:
        if cfg.get("ctc_layer", 0) > 0:
            enc.ctc_compress_method = getattr(ct.CTCCompressStrategy, s)
        out = R.run_reference_encoder(enc, x, lens, return_all_hiddens=True)
        fx["outputs"][s] = out_to_dict(out)
    return fx


def ctc_fixture():
    """Reference ``average_same_ctc_features`` on its own, incl. the SURVEY 3.5 KAT."""
    ct = R.load()
    cases = []
    g = torch.Generator().manual_seed(11)

    class Stub:  # only the attributes average_same_ctc_features touches
        pass

    def run(x, logits, lengths, strategy):
        stub = Stub()
        stub.ctc_fc = lambda _x: logits
        stub.ctc_compress_method = getattr(ct.CTCCompressStrategy, strategy)
        import warnings
        with torch.no_grad(), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            x_ctc, out, new_len = ct.ConvolutionalTransformerEncoder.average_same_ctc_features(
                stub, x, lengths)
        return out, new_len

    # KAT (SURVEY 3.5): V=4, T'=6, B=2, lens [6,4]
    V, T, B, D = 4, 6, 2, 8
    lab = torch.tensor([[2, 2, 1, 1, 1, 3], [0, 0, 0, 2, 1, 1]]).t()
    mar = torch.tensor([[1, 2, .5, 1.5, 3, 1], [2, 1, .5, 4, 9, 9]]).t()
    logits = torch.zeros(T, B, V)
    logits.scatter_(2, lab.unsqueeze(-1), mar.unsqueeze(-1))
    x = torch.randn(T, B, D, generator=g)
    lengths = torch.tensor([6, 4])
    for s in ("avg", "weighted", "softmax"):
        out, nl = run(x, logits, lengths, s)
        cases.append(dict(name="kat_" + s, strategy=s, x=x, logits=logits, lengths=lengths,
                          out=out, new_lengths=nl))
    # random run-structured cases
    for ci, (T, B, V, D, lens) in enumerate([
            (37, 3, 50, 64, [37, 20, 1]),
            (64, 4, 301, 128, [64, 64, 63, 2]),
            (5, 1, 7, 32, [5])]):
        labels = O.synthetic_ctc_bump(T, B, V, seed=100 + ci)
        logits = torch.randn(T, B, V, generator=g)
        logits = O.bump_hook(labels, 6.0)(logits)
        x = torch.randn(T, B, D, generator=g)
        lengths = torch.tensor(lens)
        for s in ("avg", "weighted", "softmax"):
            out, nl = run(x, logits, lengths, s)
            cases.append(dict(name="rand%d_%s" % (ci, s), strategy=s, x=x, logits=logits,
                              lengths=lengths, out=out, new_lengths=nl))
    return cases


def cmvn_fixture():
    R.load()
    from examples.speech_recognition.data.data_utils import apply_mv_norm
    g = torch.Generator().manual_seed(5)
    cases = []
    for T, Fd in [(50, 40), (333, 80), (2, 40)]:
        x = torch.randn(T, Fd, generator=g) * 3 + 1.5
        cases.append(dict(x=x, y=apply_mv_norm(x)))
    x = torch.randn(20, 40, generator=g)
    x[:, 3] = 0.25  # constant feature -> var < eps branch (data_utils.py:17-18)
    cases.append(dict(x=x, y=apply_mv_norm(x)))
    return cases


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    golden.save(encoder_fixture(TINY, [61, 47, 30], 0, ["avg", "weighted", "softmax"]),
                os.path.join(GOLDEN_DIR, "enc_tiny_log.pt"))
    golden.save(encoder_fixture(TINY_NOPEN, [40, 40], 1, ["avg"]),
                os.path.join(GOLDEN_DIR, "enc_tiny_nopen.pt"))
    torch.save(ctc_fixture(), os.path.join(GOLDEN_DIR, "ctc_compress.pt"))
    torch.save(cmvn_fixture(), os.path.join(GOLDEN_DIR, "cmvn.pt"))
    for f in sorted(os.listdir(GOLDEN_DIR)):
        print(f, os.path.getsize(os.path.join(GOLDEN_DIR, f)))


if __name__ == "__main__":
    main()
