"""GPU parity of the fp32 decode path (``CrossAttention.precision = "fp32"``): fbkst_xattn_fwd_f32 against fp64
on the same fp32 operands, and the module against the live-reference golden vectors and the oracle at 1e-3 under
both readings of tests/helpers.py.  An operand left in bf16 would show at the bf16 kernel's ~4e-3 output rounding,
so 1e-3 catches one.  The bf16 path must stay bit-identical around fp32 calls."""
import os

import pytest
import torch

from fbkst_b200 import ops
from fbkst_b200.cross_attention import CrossAttention, reorder_tagged
from helpers import elementwise_err, rel_err
from oracle import cross_attention_oracle as X  # checker only
from oracle.golden import load as load_golden

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-3


def _ref_core64(q, kv, mask, row_map, S, U, bsz, tgt, H):
    """fp64 attention core on the fp32 operands: (out [tgt*bsz, D], per-head weights [H, bsz, tgt, S])."""
    D = 64 * H
    rm = row_map.long().cpu()
    qd = q.double().cpu().view(tgt, bsz, H, 64)
    k = kv.double().cpu()[:, :, :D].view(S, U, H, 64)[:, rm]
    v = kv.double().cpu()[:, :, D:].view(S, U, H, 64)[:, rm]
    s = torch.einsum("tbhd,sbhd->hbts", qd, k)
    if mask is not None:
        s = s.masked_fill(mask.cpu()[rm].view(1, bsz, 1, S), float("-inf"))
    p = torch.softmax(s, dim=-1)
    return torch.einsum("hbts,sbhd->tbhd", p, v).reshape(tgt * bsz, D), p


@pytest.mark.parametrize("S,U,bsz,tgt,H,masked", [
    (1, 1, 1, 1, 2, False), (45, 3, 7, 1, 2, True), (95, 64, 320, 1, 8, True), (64, 4, 4, 5, 4, False),
    (1500, 2, 6, 1, 16, True), (333, 5, 5, 3, 8, True)])
def test_kernel_matches_fp64_on_same_operands(S, U, bsz, tgt, H, masked):
    g = torch.Generator().manual_seed(S * 31 + bsz)
    D = 64 * H
    q = (torch.randn(tgt * bsz, D, generator=g) * 0.5).to(DEV)
    kv = torch.randn(S, U, 2 * D, generator=g).to(DEV)
    row_map = torch.randint(0, U, (bsz,), generator=g).int().to(DEV)
    mask = None
    if masked:
        lens = torch.randint(1, S + 1, (U,), generator=g)
        lens[0] = S
        mask = (torch.arange(S)[None, :] >= lens[:, None]).to(DEV)
    ref_o, ref_p = _ref_core64(q, kv, mask, row_map, S, U, bsz, tgt, H)
    worst_o = worst_w = 0.0
    for mode in (0, 1, 2):
        out, w = ops.xattn_f32(q, kv, mask, row_map, S, U, bsz, tgt, H, weights=mode)
        assert out.dtype == torch.float32
        err = (out.double().cpu() - ref_o).abs().max().item() / ref_o.abs().max().item()
        assert err <= 1e-5, "out max-normalised err %g" % err
        worst_o = max(worst_o, err)
        if mode == 0:
            assert w is None
            continue
        ref_w = ref_p.mean(0) if mode == 1 else ref_p
        werr = (w.double().cpu() - ref_w).abs().max().item()
        assert werr <= 1e-6, "weights abs err %g (mode %d)" % (werr, mode)
        worst_w = max(worst_w, werr)
        if mask is not None:
            km = mask[row_map.long()].view(bsz, 1, S).expand(bsz, tgt, S)
            assert (w.masked_select(km if mode == 1 else km.expand(H, bsz, tgt, S)) == 0).all()
    print("xattn_f32 vs fp64 S=%d H=%d: out max-normalised %.3g, weights abs %.3g" % (S, H, worst_o, worst_w))


def test_out_of_range_row_map_gives_zero_rows():
    H, S, U, bsz = 2, 20, 2, 4
    q = torch.randn(bsz, 128, device=DEV)
    kv = torch.randn(S, U, 256, device=DEV)
    row_map = torch.tensor([0, 5, -1, 1], dtype=torch.int32, device=DEV)
    out, w = ops.xattn_f32(q, kv, None, row_map, S, U, bsz, 1, H, weights=1)
    assert (out[1] == 0).all() and (out[2] == 0).all() and (w[1] == 0).all() and (w[2] == 0).all()
    assert out[0].abs().sum() > 0 and abs(w[3].sum().item() - 1) < 1e-6


def test_bad_arguments_raise():
    q = torch.zeros(2, 128, device=DEV)
    kv = torch.zeros(4, 2, 256, device=DEV)
    rm = torch.zeros(2, dtype=torch.int32, device=DEV)
    with pytest.raises(ValueError):
        ops.xattn_f32(q, kv, None, rm, 5, 2, 2, 1, 2)  # S mismatch
    with pytest.raises(ValueError):
        ops.xattn_f32(q, kv, None, rm, 4, 2, 3, 1, 2)  # row_map / bsz mismatch
    with pytest.raises(ValueError):
        ops.xattn_f32(q.bfloat16(), kv, None, rm, 4, 2, 2, 1, 2)
    with pytest.raises(ValueError):
        ops.xattn_f32(q, kv.bfloat16(), None, rm, 4, 2, 2, 1, 2)


@pytest.fixture(scope="module")
def golden(golden_dir):
    return load_golden(os.path.join(golden_dir, "xattn.pt"))


def _module(c, precision="fp32"):
    m = CrossAttention(c["D"], c["H"], kdim=c["kdim"], vdim=c["kdim"]).eval()
    m.load_state_dict(c["params"], strict=True)
    m.precision = precision
    return m.to(DEV)


def _check(a, w, want_a, want_w, what):
    assert a.dtype == torch.float32 and a.shape == want_a.shape and w.shape == want_w.shape, what
    r, e = rel_err(a, want_a), elementwise_err(a, want_a)
    assert r <= TOL and e <= TOL, "%s: max-normalised %g, element-wise %g" % (what, r, e)
    assert (w.cpu() - want_w).abs().max().item() <= 1e-4 * want_w.max().item(), what
    return r, e


@pytest.mark.parametrize("lazy", [False, True])
def test_module_matches_live_reference_golden(golden, lazy):
    """Teacher-forced call, then incremental decoding as SequenceGenerator drives it (x beam replication,
    per-step reorders, finished hypotheses leaving the batch), all in fp32.  K/V cached ONCE per utterance."""
    worst = [0.0, 0.0]
    for name, c in golden.items():
        m = _module(c)
        enc = c["encoder_out"].to(DEV)
        mask = None if c["encoder_padding_mask"] is None else c["encoder_padding_mask"].to(DEV)
        U, beam, S, D = len(c["lens"]), c["beam"], c["S"], c["D"]
        a, w = m(c["full"]["query"].to(DEV), enc, enc, key_padding_mask=mask, static_kv=True,
                 need_weights=True, need_head_weights=c["need_head_weights"])
        worst = [max(x, y) for x, y in zip(worst, _check(a, w, c["full"]["attn"], c["full"]["weights"],
                                                        name + " full"))]
        order0 = torch.arange(U).view(-1, 1).repeat(1, beam).view(-1).to(DEV)
        memo = {}
        eo = reorder_tagged(enc, 1, order0, lazy, memo)
        em = None if mask is None else reorder_tagged(mask, 0, order0, lazy, memo)
        inc = {}
        rows = order0.cpu()
        for i, st in enumerate(c["steps"]):
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
            worst = [max(x, y) for x, y in zip(worst, _check(a, w, st["attn"], st["weights"],
                                                            "%s step %d" % (name, i)))]
            buf = m._get_input_buffer(inc)
            assert tuple(buf["fbkst_kv"].shape) == (S, U, 2 * D) and buf["fbkst_kv"].dtype == torch.float32
            assert buf["fbkst_row_map"].cpu().tolist() == rows.tolist()
    print("fp32 module vs live reference (lazy=%s): max-normalised %.3g, element-wise %.3g" % (lazy, *worst))


def test_module_untagged_key_and_oracle_random():
    """A caller that replicates the encoder output itself (no tags): U = bsz, identity row map."""
    g = torch.Generator().manual_seed(11)
    D, H, S, bsz = 512, 8, 95, 10
    P = X.init_params(D, D, 5)
    m = CrossAttention(D, H).eval()
    m.load_state_dict(P)
    m.precision = "fp32"
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
    _check(a, w, ra, rw, "first step")
    q2 = torch.randn(1, bsz, D, generator=g)
    ra, rw = X.cross_attention(P, H, q2, None, None, st)
    a, w = m(q2.to(DEV), None, None, incremental_state=inc, static_kv=True)  # cached: key ignored
    _check(a, w, ra, rw, "cached step")


def test_bf16_path_unaffected_and_cache_precision_is_checked():
    g = torch.Generator().manual_seed(3)
    D, H, S, bsz = 256, 4, 40, 6
    m = CrossAttention(D, H).eval()
    m.load_state_dict(X.init_params(D, D, 9))
    m = m.to(DEV)
    enc = torch.randn(S, bsz, D, generator=g).to(DEV)
    q = torch.randn(2, bsz, D, generator=g).to(DEV)
    a0, w0 = m(q, enc, enc, static_kv=True)
    m.precision = "fp32"
    a32, _ = m(q, enc, enc, static_kv=True)
    m.precision = "bf16"
    a1, w1 = m(q, enc, enc, static_kv=True)
    assert torch.equal(a0, a1) and torch.equal(w0, w1)
    assert not torch.equal(a0, a32)
    # a live incremental cache is only valid under the precision it was built with, in both directions
    q1 = q[:1]
    for built, other in (("bf16", "fp32"), ("fp32", "bf16")):
        m.precision = built
        inc = {}
        m(q1, enc, enc, incremental_state=inc, static_kv=True)
        m(q1, None, None, incremental_state=inc, static_kv=True)
        m.precision = other
        with pytest.raises(RuntimeError, match="precision"):
            m(q1, None, None, incremental_state=inc, static_kv=True)
    m.precision = "bf16"
    a2, w2 = m(q, enc, enc, static_kv=True)
    assert torch.equal(a0, a2) and torch.equal(w0, w2)


def test_half_model_gives_fp16_within_fp16_rounding_of_fp32():
    """model.half(): fp16 query and keys are upcast, the output is rounded back to fp16 once."""
    g = torch.Generator().manual_seed(5)
    D, H, S, bsz = 256, 4, 33, 5
    m16 = CrossAttention(D, H).eval()
    m16.load_state_dict(X.init_params(D, D, 13))
    m16.precision = "fp32"
    m16 = m16.to(DEV).half()
    m32 = CrossAttention(D, H).eval()  # the same fp16-valued parameters, held in fp32
    m32.load_state_dict({k: v.float() for k, v in m16.state_dict().items()})
    m32.precision = "fp32"
    m32 = m32.to(DEV)
    enc = torch.randn(S, bsz, D, generator=g).half().to(DEV)
    mask = torch.zeros(bsz, S, dtype=torch.bool, device=DEV)
    mask[1, 20:] = True
    q = torch.randn(1, bsz, D, generator=g).half().to(DEV)
    a16, _ = m16(q, enc, enc, key_padding_mask=mask, static_kv=True)
    a32, _ = m32(q.float(), enc.float(), enc.float(), key_padding_mask=mask, static_kv=True)
    assert a16.dtype == torch.float16 and a32.dtype == torch.float32
    assert ((a16.float() - a32).abs() <= a32.abs() * 2.0 ** -11 + 2.0 ** -25).all()
