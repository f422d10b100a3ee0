"""Regenerate ``tests/golden/xattn.pt`` from the LIVE reference -- TEST INFRASTRUCTURE ONLY.

    python -m oracle.make_golden_xattn

Drives the reference's own ``MultiheadAttention(encoder_decoder_attention=True)``
(fairseq/modules/multihead_attention.py) the way ``TransformerDecoderLayer.forward`` (:339-348) and
``SequenceGenerator`` (fairseq/sequence_generator.py:193-198, :255-258) do: encoder output replicated
x beam through the reference encoder's ``reorder_encoder_out`` logic, then incremental steps with
``reorder_incremental_state`` (same-size reorders and a shrinking batch).  Needs ``/root/reference``.
"""
import os

import torch

from . import cross_attention_oracle as X
from . import golden, ref_loader

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden",
                      "xattn.pt")


def run_case(mha_cls, seed, D, H, kdim, S, lens, beam, steps, need_head_weights):
    g = torch.Generator().manual_seed(seed)
    P = X.init_params(D, kdim, seed + 100)
    m = mha_cls(D, H, kdim=kdim, vdim=kdim, encoder_decoder_attention=True).eval()
    m.load_state_dict(P, strict=True)
    U = len(lens)
    enc = torch.randn(S, U, kdim, generator=g)
    mask = torch.zeros(U, S, dtype=torch.bool)
    for u, n in enumerate(lens):
        mask[u, n:] = True
    if not mask.any():
        mask = None
    case = dict(D=D, H=H, kdim=kdim, S=S, lens=lens, beam=beam, params=P, encoder_out=enc,
                encoder_padding_mask=mask, need_head_weights=need_head_weights, steps=[])
    with torch.no_grad():
        # teacher-forced (non-incremental) call, tgt_len 3  (static_kv=True, no incremental_state)
        q3 = torch.randn(3, U, D, generator=g)
        a, w = m(query=q3, key=enc, value=enc, key_padding_mask=mask, incremental_state=None,
                 static_kv=True, need_weights=True, need_head_weights=need_head_weights)
        case["full"] = dict(query=q3, attn=a, weights=w)
        # incremental generation
        order0 = torch.arange(U).view(-1, 1).repeat(1, beam).view(-1)
        eo, em = X.reorder_encoder_out(enc, mask, order0)  # same gather as conv_transformer.py:329-338
        inc = {}
        bsz = U * beam
        for si, new_order in enumerate(steps):
            if new_order is not None:
                new_order = torch.tensor(new_order, dtype=torch.long)
                m.reorder_incremental_state(inc, new_order)
                eo, em = X.reorder_encoder_out(eo, em, new_order)
                bsz = new_order.numel()
            q = torch.randn(1, bsz, D, generator=g)
            a, w = m(query=q, key=eo, value=eo, key_padding_mask=em, incremental_state=inc,
                     static_kv=True, need_weights=True, need_head_weights=need_head_weights)
            case["steps"].append(dict(new_order=new_order, query=q, attn=a, weights=w))
    return case


def main():
    ref_loader.load()
    from fairseq.modules.multihead_attention import MultiheadAttention
    cases = {
        # 3 utterances x beam 2: same-size reorders, then hypotheses of utterance 1 finish (shrink)
        "beam2_shrink": run_case(MultiheadAttention, 1, 128, 2, 128, 37, [37, 20, 9], 2,
                                 [None, [1, 0, 2, 2, 5, 4], [0, 0, 3, 2, 4, 4], [0, 1, 4, 5], [1, 1, 3, 2]],
                                 False),
        # no padding at all (mask None), kdim != D, per-head weights
        "nomask_heads": run_case(MultiheadAttention, 2, 256, 4, 192, 64, [64, 64], 3,
                                 [None, [2, 1, 0, 3, 3, 4], [0, 1, 2]], True),
        # one utterance, beam 5, src_len not a multiple of 8 / 32
        "single_beam5": run_case(MultiheadAttention, 3, 128, 2, 128, 45, [45], 5,
                                 [None, [4, 3, 2, 1, 0], [0, 0, 0, 1, 1]], False),
    }
    for p in golden.save(cases, GOLDEN):
        print("wrote", p, os.path.getsize(p), "bytes")


if __name__ == "__main__":
    main()
