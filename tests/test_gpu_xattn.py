"""GPU parity of the N4 row: fbkst_xattn_fwd through the C ABI against a torch fp32 restatement on the
SAME bf16 operands (kernel-level), and CrossAttention against the oracle / the live-reference golden
vectors through incremental decoding with beam replication, reorders and a shrinking batch.
Tolerance: bf16 path, 2e-2 relative (BASELINE.json north_star); row maps and cached shapes exact."""
import os

import pytest
import torch

from fbkst_b200 import ops
from fbkst_b200.cross_attention import CrossAttention, reorder_tagged
from oracle import cross_attention_oracle as X  # checker only
from oracle.golden import load as load_golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _ref_core(q, kv, mask, row_map, S, U, bsz, tgt, H):
    """fp32 attention core on the bf16 operands: returns (out [tgt*bsz, D], per-head weights)."""
    D = 64 * H
    qf = q.float().view(tgt, bsz, H, 64)
    k = kv.float()[:, :, :D].view(S, U, H, 64)[:, row_map.long()]  # [S, bsz, H, 64]
    v = kv.float()[:, :, D:].view(S, U, H, 64)[:, row_map.long()]
    s = torch.einsum("tbhd,sbhd->hbts", qf, k)
    if mask is not None:
        s = s.masked_fill(mask[row_map.long()].view(1, bsz, 1, S), float("-inf"))
    p = torch.softmax(s, dim=-1)
    o = torch.einsum("hbts,sbhd->tbhd", p, v).reshape(tgt * bsz, D)
    return o, p


@pytest.mark.parametrize("S,U,bsz,tgt,H,masked", [
    (1, 1, 1, 1, 2, False), (45, 3, 7, 1, 2, True), (95, 64, 320, 1, 8, True), (64, 4, 4, 5, 4, False),
    (1500, 2, 6, 1, 16, True), (333, 5, 5, 3, 8, True)])
def test_kernel_matches_fp32_on_same_operands(S, U, bsz, tgt, H, masked):
    g = torch.Generator().manual_seed(S * 31 + bsz)
    D = 64 * H
    q = (torch.randn(tgt * bsz, D, generator=g) * 0.5).bfloat16().to(DEV)
    kv = torch.randn(S, U, 2 * D, generator=g).bfloat16().to(DEV)
    row_map = torch.randint(0, U, (bsz,), generator=g).int().to(DEV)
    mask = None
    if masked:
        lens = torch.randint(1, S + 1, (U,), generator=g)
        lens[0] = S
        mask = (torch.arange(S)[None, :] >= lens[:, None]).to(DEV)
    for mode in (0, 1, 2):
        out, w = ops.xattn(q, kv, mask, row_map, S, U, bsz, tgt, H, weights=mode)
        ref_o, ref_p = _ref_core(q, kv, mask, row_map, S, U, bsz, tgt, H)
        err = (out.float() - ref_o).abs().max().item() / ref_o.abs().max().item()
        assert err < 8e-3, "out rel err %g (bf16 output rounding is 4e-3)" % err
        if mode == 1:
            assert (w - ref_p.mean(0)).abs().max().item() < 1e-5
            if mask is not None:
                assert (w.masked_select(mask[row_map.long()].view(bsz, 1, S).expand(bsz, tgt, S)) == 0).all()
        elif mode == 2:
            assert (w - ref_p).abs().max().item() < 1e-5
        else:
            assert w is None


def test_out_of_range_row_map_gives_zero_rows():
    H, S, U, bsz = 2, 20, 2, 4
    q = torch.randn(bsz, 128).bfloat16().to(DEV)
    kv = torch.randn(S, U, 256).bfloat16().to(DEV)
    row_map = torch.tensor([0, 5, -1, 1], dtype=torch.int32, device=DEV)
    out, w = ops.xattn(q, kv, None, row_map, S, U, bsz, 1, H, weights=1)
    assert (out[1] == 0).all() and (out[2] == 0).all() and (w[1] == 0).all() and (w[2] == 0).all()
    assert out[0].abs().sum() > 0 and abs(w[3].sum().item() - 1) < 1e-5


def test_bad_arguments_raise():
    q = torch.zeros(2, 128, dtype=torch.bfloat16, device=DEV)
    kv = torch.zeros(4, 2, 256, dtype=torch.bfloat16, device=DEV)
    rm = torch.zeros(2, dtype=torch.int32, device=DEV)
    with pytest.raises(ValueError):
        ops.xattn(q, kv, None, rm, 5, 2, 2, 1, 2)  # S mismatch
    with pytest.raises(ValueError):
        ops.xattn(q.float(), kv, None, rm, 4, 2, 2, 1, 2)


@pytest.fixture(scope="module")
def golden(golden_dir):
    return load_golden(os.path.join(golden_dir, "xattn.pt"))


def _module(c):
    m = CrossAttention(c["D"], c["H"], kdim=c["kdim"], vdim=c["kdim"]).eval()
    m.load_state_dict(c["params"], strict=True)
    return m.to(DEV)


def _rel(a, b):
    return ((a.float().cpu() - b).abs().max() / b.abs().max()).item()


@pytest.mark.parametrize("lazy", [False, True])
def test_module_matches_live_reference_golden(golden, lazy):
    """Incremental decoding as SequenceGenerator drives it: x beam replication, per-step reorders,
    finished hypotheses leaving the batch.  K/V must be cached ONCE per utterance."""
    for name, c in golden.items():
        m = _module(c)
        enc = c["encoder_out"].to(DEV)
        mask = None if c["encoder_padding_mask"] is None else c["encoder_padding_mask"].to(DEV)
        U, beam, S, D = len(c["lens"]), c["beam"], c["S"], c["D"]
        # teacher-forced call (no incremental state, tgt_len 3)
        a, w = m(c["full"]["query"].to(DEV), enc, enc, key_padding_mask=mask, static_kv=True,
                 need_weights=True, need_head_weights=c["need_head_weights"])
        assert _rel(a, c["full"]["attn"]) < 2e-2, name
        assert (w.cpu() - c["full"]["weights"]).abs().max().item() < 2e-2 * c["full"]["weights"].max().item()
        order0 = torch.arange(U).view(-1, 1).repeat(1, beam).view(-1).to(DEV)
        memo = {}
        eo = reorder_tagged(enc, 1, order0, lazy, memo)
        em = None if mask is None else reorder_tagged(mask, 0, order0, lazy, memo)
        inc = {}
        rows = order0.cpu()
        for st in c["steps"]:
            if st["new_order"] is not None:
                no = st["new_order"].to(DEV)
                m.reorder_incremental_state(inc, no)
                memo = {}
                eo = reorder_tagged(eo, 1, no, lazy, memo)
                em = None if em is None else reorder_tagged(em, 0, no, lazy, memo)
                if st["new_order"].numel() != rows.numel():
                    rows = rows[st["new_order"]]
            a, w = m(st["query"].to(DEV), eo, eo, key_padding_mask=em, incremental_state=inc,
                     static_kv=True, need_weights=True, need_head_weights=c["need_head_weights"])
            assert a.shape == st["attn"].shape and w.shape == st["weights"].shape
            assert _rel(a, st["attn"]) < 2e-2, name
            assert (w.cpu() - st["weights"]).abs().max().item() < 2e-2 * st["weights"].max().item()
            buf = m._get_input_buffer(inc)
            assert tuple(buf["fbkst_kv"].shape) == (S, U, 2 * D)  # once per utterance, never x beam
            assert buf["fbkst_row_map"].cpu().tolist() == rows.tolist()


def test_module_untagged_key_and_oracle_random():
    """A caller that replicates the encoder output itself (no tags): U = bsz, identity row map."""
    g = torch.Generator().manual_seed(11)
    D, H, S, bsz = 512, 8, 95, 10
    P = X.init_params(D, D, 5)
    m = CrossAttention(D, H).eval()
    m.load_state_dict(P)
    m = m.to(DEV)
    enc = torch.randn(S, bsz, D, generator=g)
    mask = torch.zeros(bsz, S, dtype=torch.bool)
    mask[3, 40:] = True
    mask[7, 1:] = True
    q = torch.randn(1, bsz, D, generator=g)
    st = {}
    ra, rw = X.cross_attention(P, H, q, enc, mask, st)
    inc = {}
    a, w = m(q.to(DEV), enc.to(DEV), enc.to(DEV), key_padding_mask=mask.to(DEV), incremental_state=inc,
             static_kv=True)
    assert _rel(a, ra) < 2e-2 and (w.cpu() - rw).abs().max().item() < 2e-2
    q2 = torch.randn(1, bsz, D, generator=g)
    ra, rw = X.cross_attention(P, H, q2, None, None, st)
    a, w = m(q2.to(DEV), None, None, incremental_state=inc, static_kv=True)  # cached: key ignored
    assert _rel(a, ra) < 2e-2 and (w.cpu() - rw).abs().max().item() < 2e-2
