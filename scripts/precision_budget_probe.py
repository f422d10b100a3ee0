"""Operand-precision budget of the fp32 path, emulated on the CPU oracle (DESIGN section F, error table).

Every GEMM / convolution / attention-product operand of oracle/encoder_oracle.py is rounded as a tensor core
would see it, with fp32 accumulation, and the output is compared with the unrounded fp32 oracle under both
readings of tests/helpers.parity_report:

    plain-rn     TF32 operands, round to nearest
    plain-trunc  TF32 operands, truncated (what the tensor core does to unrounded fp32)
    split        hi = tf32_rn(x), lo = tf32_rn(x - hi), hi.hi + hi.lo + lo.hi (the kernels of tf32x3.cu)

    python scripts/precision_budget_probe.py [--config cfg1|cfg2] [--utts N]
"""
import argparse
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "fbk-fairseq-st_b200")]
from helpers import parity_report  # noqa: E402
from oracle import encoder_oracle as O  # noqa: E402


def tf32_rn(t):
    i = t.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)  # round half away on the 13 dropped bits


def tf32_trunc(t):
    return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


def products(mode):
    """(a, b) -> list of (a_i, b_i) operand pairs whose products are summed in fp32."""
    if mode == "plain-rn":
        return lambda a, b: [(tf32_rn(a), tf32_rn(b))]
    if mode == "plain-trunc":
        return lambda a, b: [(tf32_trunc(a), tf32_trunc(b))]

    def split(a, b):
        ah, bh = tf32_rn(a), tf32_rn(b)
        al, bl = tf32_rn(a - ah), tf32_rn(b - bh)
        return [(al, bh), (ah, bl), (ah, bh)]
    return split


def patched(mode):
    pairs = products(mode)
    lin, bmm, conv = F.linear, torch.bmm, F.conv2d

    def linear(x, w, b=None):
        y = sum(lin(p, q) for p, q in pairs(x, w))
        return y if b is None else y + b

    def bmm_(a, b):
        return sum(bmm(p, q) for p, q in pairs(a, b))

    def conv2d(x, w, b=None, *args, **kw):
        y = sum(conv(p, q, None, *args, **kw) for p, q in pairs(x, w))
        return y if b is None else y + b[None, :, None, None]
    return linear, bmm_, conv2d, (lin, bmm, conv)


def run(mode, sd, cfg, x, lens):
    if mode is None:
        return O.encoder_forward(sd, cfg, x, lens)
    linear, bmm_, conv2d, orig = patched(mode)
    F.linear, torch.bmm, F.conv2d = linear, bmm_, conv2d
    try:
        return O.encoder_forward(sd, cfg, x, lens)
    finally:
        F.linear, torch.bmm, F.conv2d = orig


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="cfg1", choices=["cfg1", "cfg2"])
    ap.add_argument("--utts", type=int, default=None, help="utterances (default 8 for cfg1, 4 for cfg2)")
    args = ap.parse_args()
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    if args.config == "cfg1":  # bench.py cfg1: 6L d256, no penalty, compression avg @4, 8 x 1000 .. 400
        cfg = dict(embed_dim=256, ffn_dim=768, heads=4, layers=6, conv_channels=64, feat_dim=40, vocab=105,
                   distance_penalty=None, ctc_layer=4, ctc_strategy="avg")
        lengths = [1000, 950, 900, 800, 700, 600, 500, 400][: args.utts or 8]
    else:  # cfg2-like: 11L d512, log penalty, compression avg @8, utterances up to 1500 frames
        cfg = dict(embed_dim=512, ffn_dim=2048, heads=8, layers=11, conv_channels=64, feat_dim=40, vocab=8005,
                   distance_penalty="log", ctc_layer=8, ctc_strategy="avg")
        lengths = [1500, 1333, 1001, 777][: args.utts or 4]
    sd = O.init_state_dict(cfg, seed=1)
    x, lens = O.synthetic_batch(lengths, cfg["feat_dim"], seed=77)
    ref = run(None, sd, cfg, x, lens)
    nl = ref["src_lengths"].tolist()
    print("%s, %d utterances, random-init weights" % (args.config, len(lengths)))
    print("%-12s %12s %12s" % ("operands", "max-norm", "element-wise"))
    for mode in ("plain-rn", "plain-trunc", "split"):
        out = run(mode, sd, cfg, x, lens)
        if out["src_lengths"].tolist() != nl:
            print("%-12s compressed lengths differ from the fp32 oracle" % mode)
            continue
        rep = parity_report(out["encoder_out"], ref["encoder_out"], nl)
        print("%-12s %12.2e %12.2e" % (mode, rep["max_rel"], rep["elementwise"]))


if __name__ == "__main__":
    main()
