"""GPU parity of the decoder self-attention (N5): fbkst_dec_self_attn_fwd / _f32 against fp64 on the same operands
(ancestry gathers, per-step padding, incremental / full / causal modes, all weight modes), and DecoderSelfAttention
against the oracle through beam reorders and a shrinking batch, under both readings of tests/helpers.py."""
import pytest
import torch

from fbkst_b200 import ops
from fbkst_b200.self_attention import DecoderSelfAttention
from helpers import TOL_BF16, elementwise_err, rel_err
from oracle import self_attention_oracle as SA  # checker only

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL_F32 = 1e-3


def _ref_core64(q, cache, anc, pad, n_keys, bsz, tgt, H, causal):
    """fp64 core on the kernel's operands: (out [tgt*bsz, D], per-head weights [H, bsz, tgt, n_keys]).  A key whose
    ancestry entry is out of range is masked; a query with no visible unmasked key gets zeros."""
    D = 64 * H
    c = cache.double().cpu()
    R = c.shape[1]
    steps = torch.arange(n_keys)[:, None].expand(n_keys, bsz)
    rows = torch.arange(bsz)[None, :].expand(n_keys, bsz) if anc is None else anc[:n_keys].long().cpu()
    bad = (rows < 0) | (rows >= R)
    rows = rows.clamp(0, R - 1)
    k = c[steps, rows, D:2 * D].view(n_keys, bsz, H, 64)
    v = c[steps, rows, 2 * D:].view(n_keys, bsz, H, 64)
    masked = bad if pad is None else bad | pad.cpu()[steps, rows].bool()  # [n_keys, bsz]
    s = torch.einsum("tbhd,sbhd->hbts", q.double().cpu().view(tgt, bsz, H, 64), k)
    s = s.masked_fill(masked.t().reshape(1, bsz, 1, n_keys), float("-inf"))
    if causal:
        s = s.masked_fill(torch.ones(tgt, n_keys).triu(1).bool().view(1, 1, tgt, n_keys), float("-inf"))
    p = torch.softmax(s, dim=-1).nan_to_num(0.0)
    return torch.einsum("hbts,sbhd->tbhd", p, v).reshape(tgt * bsz, D), p


def _check_kernel(dtype, q, cache, anc, pad, n_keys, bsz, tgt, H, mode):
    fn = ops.dec_self_attn_f32 if dtype == torch.float32 else ops.dec_self_attn
    ref_o, ref_p = _ref_core64(q, cache, anc, pad, n_keys, bsz, tgt, H, mode == ops.SA_CAUSAL)
    tol_o, tol_w = (1e-5, 1e-6) if dtype == torch.float32 else (8e-3, 1e-5)
    worst = [0.0, 0.0]
    for wm in (0, 1, 2):
        out, w = fn(q, cache, anc, pad, n_keys, bsz, tgt, H, mode=mode, weights=wm)
        assert out.dtype == dtype and out.shape == (tgt * bsz, 64 * H)
        err = (out.double().cpu() - ref_o).abs().max().item() / ref_o.abs().max().item()
        assert err <= tol_o, "out max-normalised err %g (weights mode %d)" % (err, wm)
        worst[0] = max(worst[0], err)
        if wm == 0:
            assert w is None
            continue
        ref_w = ref_p.mean(0) if wm == 1 else ref_p
        werr = (w.double().cpu() - ref_w).abs().max().item()
        assert werr <= tol_w, "weights abs err %g (mode %d)" % (werr, wm)
        worst[1] = max(worst[1], werr)
        zero = ref_w == 0  # masked, out-of-range and future keys: exactly 0
        assert (w.cpu()[zero] == 0).all()
    return worst


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("H", [8, 16])
@pytest.mark.parametrize("t", [1, 2, 63, 64, 65, 300])
def test_incremental_kernel_matches_fp64(dtype, H, t):
    """One query per hypothesis over steps 0..t-1, keys gathered through a random ancestry table (with two
    out-of-range entries), random per-step padding bytes; q both as a separate tensor and as the cache's view."""
    g = torch.Generator().manual_seed(t * 131 + H)
    D, R, bsz = 64 * H, 12, 10
    cache = torch.randn(t + 3, R, 3 * D, generator=g)
    cache[..., :D] *= 0.125  # the q columns hold pre-scaled queries, as the projection writes them
    cache = cache.to(dtype).to(DEV)
    anc = torch.randint(0, R, (t, bsz), generator=g, dtype=torch.int32)
    anc[-1] = torch.arange(bsz, dtype=torch.int32)
    if t > 2:
        anc[1, 3], anc[2, 4] = R, -1
    pad = torch.rand(t + 3, R, generator=g) < 0.2  # t == 1: a row whose only key is padded is a zero row
    anc, pad = anc.to(DEV), pad.to(DEV)
    q_sep = (torch.randn(bsz, D, generator=g) * 0.125).to(dtype).to(DEV)
    worst = _check_kernel(dtype, q_sep, cache, anc, pad, t, bsz, 1, H, ops.SA_INCREMENTAL)
    w2 = _check_kernel(dtype, cache[t - 1, :bsz, :D], cache, anc, None, t, bsz, 1, H, ops.SA_INCREMENTAL)
    print("dec_self_attn %s H=%d t=%d: out %.3g, weights %.3g" % (dtype, H, t, max(worst[0], w2[0]),
                                                                   max(worst[1], w2[1])))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("mode", ["full", "causal"])
@pytest.mark.parametrize("T,H", [(1, 8), (37, 8), (70, 16)])
def test_full_and_causal_kernel_matches_fp64(dtype, mode, T, H):
    g = torch.Generator().manual_seed(T * 7 + H)
    D, bsz = 64 * H, 5
    cache = torch.randn(T, bsz, 3 * D, generator=g)
    cache[..., :D] *= 0.125  # pre-scaled queries
    cache = cache.to(dtype).to(DEV)
    pad = torch.zeros(T, bsz, dtype=torch.bool)
    pad[T // 2:, 1] = True  # right-padded target of row 1
    pad = pad.to(DEV)
    m = ops.SA_CAUSAL if mode == "causal" else ops.SA_FULL
    _check_kernel(dtype, cache.view(T * bsz, 3 * D)[:, :D], cache, None, pad, T, bsz, T, H, m)


def test_all_masked_query_gives_zero_row():
    H, D, bsz = 8, 512, 3
    cache = torch.randn(4, bsz, 3 * D, device=DEV)
    anc = torch.zeros(2, bsz, dtype=torch.int32, device=DEV)
    pad = torch.zeros(4, bsz, dtype=torch.uint8, device=DEV)
    pad[0, 0] = pad[1, 0] = 1
    out, w = ops.dec_self_attn_f32(cache[1, :, :D], cache, anc, pad, 2, bsz, 1, H, weights=1)
    assert (out[:] == 0).all() and (w == 0).all()  # every hypothesis reads row 0, which is padded at both steps
    anc[1] = torch.arange(bsz, dtype=torch.int32, device=DEV)
    out, w = ops.dec_self_attn_f32(cache[1, :, :D], cache, anc, pad, 2, bsz, 1, H, weights=1)
    assert (out[0] == 0).all() and (w[0] == 0).all()
    assert out[1].abs().sum() > 0 and abs(w[1].sum().item() - 1) < 1e-6 and w[1, 0, 0].item() == 0


def test_bad_arguments_raise():
    H, D, bsz = 2, 128, 3
    cache = torch.zeros(4, bsz, 3 * D, device=DEV)
    q = cache[0, :, :D]
    anc = torch.zeros(4, bsz, dtype=torch.int32, device=DEV)
    with pytest.raises(ValueError):
        ops.dec_self_attn_f32(q, cache, anc, None, 5, bsz, 1, H)  # more keys than cached steps
    with pytest.raises(ValueError):
        ops.dec_self_attn_f32(q, cache, anc[:, :2], None, 3, bsz, 1, H)  # anc for another batch size
    with pytest.raises(ValueError):
        ops.dec_self_attn_f32(q, cache, anc, torch.zeros(4, 2, dtype=torch.uint8, device=DEV), 3, bsz, 1, H)
    with pytest.raises(ValueError):
        ops.dec_self_attn_f32(q.bfloat16(), cache, anc, None, 3, bsz, 1, H)
    with pytest.raises(ValueError):
        ops.dec_self_attn(q, cache, anc, None, 3, bsz, 1, H)  # fp32 operands on the bf16 kernel
    with pytest.raises(ValueError):
        ops.dec_self_attn_f32(q, cache, anc, None, 3, bsz, 1, H, mode=3)
    with pytest.raises(ValueError, match="incremental"):  # two queries per row in incremental mode
        ops.dec_self_attn_f32(torch.zeros(2 * bsz, D, device=DEV), cache, anc, None, 3, bsz, 2, H)
    with pytest.raises(ValueError, match="n_keys == tgt_len"):
        ops.dec_self_attn_f32(torch.zeros(2 * bsz, D, device=DEV), cache, None, None, 3, bsz, 2, H, mode=ops.SA_FULL)
    with pytest.raises(ValueError, match="cache holds"):  # more hypotheses than cache rows
        ops.dec_self_attn_f32(torch.zeros(4, D, device=DEV), cache, None, None, 3, 4, 1, H)
    big = torch.zeros(17 * 64 * 3, device=DEV).view(1, 1, -1)
    with pytest.raises(ValueError, match="heads"):
        ops.dec_self_attn_f32(big[0, :, :17 * 64], big, None, None, 1, 1, 1, 17)
    long = torch.zeros(3000, 1, 3 * 1024, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(ValueError, match="shared memory"):
        ops.dec_self_attn(long[0, :, :1024], long, None, None, 3000, 1, 1, 16)


# ------------------------------------------------------------------------------------------------ module
def _module(D, H, seed, precision):
    P = SA.init_params(D, seed)
    m = DecoderSelfAttention(D, H).eval()
    m.load_state_dict(P, strict=True)
    m.precision = precision
    return m.to(DEV), {k: v.double() for k, v in P.items()}


def _check(a, want, tol, what):
    r, e = rel_err(a, want), elementwise_err(a, want)
    assert r <= tol and e <= tol, "%s: max-normalised %g, element-wise %g" % (what, r, e)
    return r, e


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_module_matches_oracle_through_reorders(precision):
    """40 decode steps as SequenceGenerator drives them: a same-size beam permutation before every step, finished
    sentences leaving the batch three times, a padded token at one step, the cache growing past its first
    capacity.  Compared with the oracle's torch.cat cache in fp64."""
    tol = TOL_BF16 if precision == "bf16" else TOL_F32
    D, H, n_sent, beam = 512, 8, 4, 5
    m, P = _module(D, H, 21, precision)
    g = torch.Generator().manual_seed(22)
    n = n_sent * beam
    inc, st = {}, {}
    worst = [0.0, 0.0]
    for t in range(40):
        if t > 0:
            if t in (6, 13, 27):  # one sentence finishes: its beam leaves the batch
                drop = torch.randint(0, n // beam, (1,), generator=g).item()
                order = torch.tensor([r for r in range(n) if r // beam != drop])
            else:
                order = torch.arange(n).view(-1, beam)
                order = order.gather(1, torch.randint(0, beam, order.shape, generator=g)).view(-1)
            m.reorder_incremental_state(inc, order.to(DEV))
            SA.reorder_state(st, order)
            n = order.numel()
        x = torch.randn(1, n, D, generator=g)
        kpm = None
        if t == 9:
            kpm = torch.zeros(n, 1, dtype=torch.bool)
            kpm[2, 0] = kpm[7, 0] = True
        want, want_w = SA.self_attention(P, H, x.double(), key_padding_mask=kpm, state=st)
        a, w = m(x.to(DEV), x.to(DEV), x.to(DEV), key_padding_mask=None if kpm is None else kpm.to(DEV),
                 incremental_state=inc, need_weights=True)
        assert a.dtype == torch.float32 and a.shape == (1, n, D) and w.shape == (n, 1, t + 1)
        worst = [max(x_, y_) for x_, y_ in zip(worst, _check(a, want, tol, "%s step %d" % (precision, t)))]
        if precision == "fp32":
            assert (w.double().cpu() - want_w).abs().max().item() <= 1e-4
        if kpm is not None:
            assert (w[kpm.view(-1).to(DEV), 0, t] == 0).all()
        buf = m._get_input_buffer(inc)
        assert buf["fbkst_steps"] == t + 1 and buf["fbkst_cache"].shape[1] == n_sent * beam
    assert buf["fbkst_cache"].shape[0] == 2 * DecoderSelfAttention.INITIAL_STEPS
    print("DecoderSelfAttention %s vs oracle over 40 steps: max-normalised %.3g, element-wise %.3g" %
          (precision, *worst))


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_full_path_equals_incremental_and_oracle(precision):
    """SequenceScorer's call: the whole target at once under fairseq's future mask (or no mask) with right
    padding, against the step-by-step outputs and the oracle.  bf16 is held to the oracle under the max-normalised
    reading here; its element-wise reading is asserted step by step in test_module_matches_oracle_through_reorders
    (the full call is checked equal to those steps)."""
    D, H, T, bsz = 512, 8, 23, 6
    m, P = _module(D, H, 31, precision)
    g = torch.Generator().manual_seed(32)
    x = torch.randn(T, bsz, D, generator=g)
    kpm = torch.zeros(bsz, T, dtype=torch.bool)
    kpm[2, 15:] = True
    fm = SA.future_mask(T)
    a, w = m(x.to(DEV), None, None, key_padding_mask=kpm.to(DEV), attn_mask=fm.to(DEV), need_weights=True)
    want, want_w = SA.self_attention(P, H, x.double(), key_padding_mask=kpm, attn_mask=fm.double())
    if precision == "fp32":
        _check(a, want, TOL_F32, "causal full call")
    else:
        assert rel_err(a, want) <= TOL_BF16, "causal full call: max-normalised %g" % rel_err(a, want)
    assert w.shape == (bsz, T, T) and (w.cpu()[want_w == 0] == 0).all()
    inc = {}
    steps = []
    for t in range(T):
        at, _ = m(x[t:t + 1].to(DEV), None, None, key_padding_mask=kpm[:, t:t + 1].to(DEV), incremental_state=inc)
        steps.append(at)
    inc_out = torch.cat(steps, 0)
    r = rel_err(a, inc_out)
    assert r <= (1e-5 if precision == "fp32" else 1e-2), "full vs incremental: %g" % r
    a0, _ = m(x.to(DEV), None, None, need_weights=False)  # no mask: every query sees every key
    want0 = SA.self_attention(P, H, x.double())[0]
    if precision == "fp32":
        _check(a0, want0, TOL_F32, "unmasked full call")
    else:
        assert rel_err(a0, want0) <= TOL_BF16, "unmasked full call: max-normalised %g" % rel_err(a0, want0)


def test_reorder_never_copies_the_cache():
    m, _ = _module(512, 8, 41, "bf16")
    g = torch.Generator().manual_seed(42)
    inc = {}
    for _ in range(5):
        m(torch.randn(1, 10, 512, generator=g).to(DEV), None, None, incremental_state=inc)
    buf = m._get_input_buffer(inc)
    cache, pad = buf["fbkst_cache"], buf["fbkst_pad"]
    # bit patterns of the whole buffer: the steps not yet written hold uninitialised memory, possibly NaNs
    bits = lambda c: c.view(torch.int16)
    ptr, snap = cache.data_ptr(), bits(cache).clone()
    for order in ([1, 0, 3, 2, 5, 4, 7, 6, 9, 8], [0, 0, 2, 2, 4, 4, 6, 6, 8, 8], [0, 1, 2, 3, 4], [4, 0]):
        m.reorder_incremental_state(inc, torch.tensor(order, device=DEV))
        buf = m._get_input_buffer(inc)
        assert buf["fbkst_cache"].data_ptr() == ptr and torch.equal(bits(buf["fbkst_cache"]), snap)
        assert buf["fbkst_pad"] is pad
    m(torch.randn(1, 2, 512, generator=g).to(DEV), None, None, incremental_state=inc)
    cache = m._get_input_buffer(inc)["fbkst_cache"]
    assert cache.data_ptr() == ptr and torch.equal(bits(cache)[:5], snap[:5])  # appended, earlier steps untouched


def test_precision_switch_with_live_cache_raises():
    m, _ = _module(256, 4, 51, "bf16")
    x = torch.randn(1, 3, 256, device=DEV)
    for built, other in (("bf16", "fp32"), ("fp32", "bf16")):
        m.precision = built
        inc = {}
        m(x, None, None, incremental_state=inc)
        m(x, None, None, incremental_state=inc)
        m.precision = other
        with pytest.raises(RuntimeError, match="precision"):
            m(x, None, None, incremental_state=inc)


def test_unsupported_masks_and_steps_raise():
    m, _ = _module(256, 4, 52, "bf16")
    x = torch.randn(4, 3, 256, device=DEV)
    with pytest.raises(NotImplementedError, match="future mask"):
        m(x, None, None, attn_mask=torch.zeros(4, 4, device=DEV) - 1.0)
    with pytest.raises(NotImplementedError, match="future mask"):
        m(x, None, None, attn_mask=SA.future_mask(4).t().contiguous().to(DEV))
    with pytest.raises(NotImplementedError):
        m(x, None, None, incremental_state={})  # four tokens in one incremental step
    with pytest.raises(NotImplementedError):
        m(x[:1], None, None, incremental_state={}, attn_mask=torch.zeros(1, 1, device=DEV))


def test_half_model_gives_fp16_within_fp16_rounding_of_fp32():
    """model.half(): fp16 queries are upcast, the output is rounded back to fp16 once."""
    g = torch.Generator().manual_seed(5)
    D, H, bsz = 256, 4, 5
    m16, _ = _module(D, H, 53, "fp32")
    m16 = m16.half()
    m32 = DecoderSelfAttention(D, H).eval()  # the same fp16-valued parameters, held in fp32
    m32.load_state_dict({k: v.float() for k, v in m16.state_dict().items()})
    m32.precision = "fp32"
    m32 = m32.to(DEV)
    inc16, inc32 = {}, {}
    for _ in range(3):
        x = torch.randn(1, bsz, D, generator=g).half().to(DEV)
        a16, _ = m16(x, None, None, incremental_state=inc16)
        a32, _ = m32(x.float(), None, None, incremental_state=inc32)
        assert a16.dtype == torch.float16 and a32.dtype == torch.float32
        assert ((a16.float() - a32).abs() <= a32.abs() * 2.0 ** -11 + 2.0 ** -25).all()


def test_bf16_outputs_bit_identical_around_fp32_calls():
    m, _ = _module(256, 4, 54, "bf16")
    g = torch.Generator().manual_seed(55)
    x = torch.randn(6, 4, 256, generator=g).to(DEV)
    fm = SA.future_mask(6).to(DEV)
    a0, w0 = m(x, None, None, attn_mask=fm)
    inc = {}
    s0, _ = m(x[:1], None, None, incremental_state=inc)
    m.precision = "fp32"
    a32, _ = m(x, None, None, attn_mask=fm)
    m(x[:1], None, None, incremental_state={})
    m.precision = "bf16"
    a1, w1 = m(x, None, None, attn_mask=fm)
    s1, _ = m(x[:1], None, None, incremental_state={})
    assert torch.equal(a0, a1) and torch.equal(w0, w1) and torch.equal(s0, s1)
    assert not torch.equal(a0, a32)
