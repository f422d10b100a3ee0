"""The fp32-accurate inference path (``encoder.precision = "fp32"``): split-TF32 tensor-core GEMM and attention,
fp32 conv front end, and the whole encoder against the fp32 oracle.

Kernels are checked against fp64 torch; the encoder against ``oracle/encoder_oracle.py`` under both readings of
tests/helpers.py at 1e-3 (the contract's "1e-3 relative under fp32 or TF32"), with lengths, masks and CTC labels
exact.  The bf16 default path must not change when another encoder switches precision."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import bench  # noqa: E402
from helpers import parity_report  # noqa: E402
from oracle import encoder_oracle as O  # noqa: E402

TOL_F32 = 1e-3
# attention against fp64: fp32 softmax sums over up to 2600 keys and ex2.approx add ~1e-5 to the split's ~1e-6
TOL_ATTN = 3e-5


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    assert torch.isfinite(a).all()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


# ----------------------------------------------------------------------------------------------- GEMM
@pytest.mark.parametrize("M,N,K", [(300, 768, 256), (1000, 105, 256), (257, 512, 2048), (129, 2048, 512),
                                   (4000, 256, 640), (77, 64, 576), (515, 1536, 512), (640, 64, 1152)])
@pytest.mark.parametrize("epi", ["bias", "relu", "residual", "affine"])
def test_linear_f32_vs_fp64(M, N, K, epi):
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(M * 7 + N + K)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / math.sqrt(K)
    b = torch.randn(N, generator=g)
    r = torch.randn(M, N, generator=g)
    sc, sh = torch.rand(N, generator=g) + 0.5, torch.randn(N, generator=g)
    ref = a.double() @ w.double().T + b.double()
    kw = {}
    if epi in ("relu", "affine"):
        ref = ref.clamp_min(0)
        kw["relu"] = True
    if epi == "affine":
        ref = ref * sc.double() + sh.double()
        kw["affine"] = (sc.cuda(), sh.cuda())
    if epi == "residual":
        ref = ref + r.double()
        kw["residual"] = r.cuda()
    out = ops.linear_f32(a.cuda(), w.cuda(), b.cuda(), **kw)
    torch.cuda.synchronize()
    assert out.shape == (M, N)
    assert _rel(out, ref) <= 1e-5


def test_linear_f32_plain_tf32_would_not_pass():
    """The split matters: the same GEMM with operands rounded to TF32 is ~100x further from fp64."""
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(3)
    a, w = torch.randn(512, 512, generator=g), torch.randn(256, 512, generator=g)
    ref = a.double() @ w.double().T
    out = ops.linear_f32(a.cuda(), w.cuda())
    tf32 = lambda t: (t.view(torch.int32) + 0x1000 & ~0x1fff).view(torch.float32)  # noqa: E731
    plain = tf32(a).double() @ tf32(w).double().T
    assert _rel(out, ref) * 30 < _rel(plain, ref)


def test_linear_f32_row_limit():
    """Rows at or beyond count * mult are neither computed nor written."""
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(5)
    M, N, K = 600, 256, 512
    a, w = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g)
    out = torch.full((M, N), 7.0, device="cuda")
    cnt = torch.tensor([37], dtype=torch.int32, device="cuda")
    ops.linear_f32(a.cuda(), w.cuda(), out=out, rows_limit=(cnt, 4))
    ref = a.double() @ w.double().T
    assert _rel(out[:148], ref[:148]) <= 1e-5
    assert bool((out[148:] == 7.0).all())


# ----------------------------------------------------------------------------------------- attention
def _attn_ref(qkv, lengths, L, B, H, log_penalty):
    D = 64 * H
    x = qkv.double().cpu().view(L, B, 3, H, 64)
    q, k, v = x[:, :, 0], x[:, :, 1], x[:, :, 2]
    s = torch.einsum("ibhd,jbhd->bhij", q, k)
    if log_penalty:
        i = torch.arange(L, dtype=torch.float64)
        s = s - torch.log((i[:, None] - i[None, :]).abs()).clamp_min(0)
    key_pad = torch.arange(L)[None, :] >= torch.tensor(lengths)[:, None]
    s = s.masked_fill(key_pad[:, None, None, :], float("-inf"))
    p = torch.softmax(s, dim=-1)
    return torch.einsum("bhij,jbhd->ibhd", p, v).reshape(L, B, D)


@pytest.mark.parametrize("L,H,log_penalty", [(250, 4, False), (375, 8, True), (375, 16, False), (1500, 8, True),
                                             (2600, 4, True), (250, 16, True)])
def test_attention_f32_vs_fp64(L, H, log_penalty):
    from fbkst_b200 import ops
    lengths = [L, L - 1, (2 * L) // 3 + 1, 65, 1][: 3 if L > 1000 else 5]
    B = len(lengths)
    g = torch.Generator().manual_seed(L + H)
    qkv = torch.randn(L * B, 3 * 64 * H, generator=g)
    qkv[:, : 64 * H] *= 0.125 * 3.0  # pre-scaled q, peaky enough that the penalty and the mask matter
    out = ops.attention_f32(qkv.cuda(), torch.tensor(lengths, dtype=torch.int32).cuda(), L, B, H, log_penalty)
    ref = _attn_ref(qkv, lengths, L, B, H, log_penalty)
    got = out.view(L, B, 64 * H).double().cpu()
    for b, n in enumerate(lengths):
        assert _rel(got[:n, b], ref[:n, b]) <= TOL_ATTN, (b, n)
        # 128-query tiles entirely beyond the length are zero
        assert bool((got[(n + 127) // 128 * 128:, b] == 0).all())


def test_attention_f32_q_limit():
    from fbkst_b200 import ops
    L, B, H = 600, 3, 8
    lengths = [180, 300, 90]
    g = torch.Generator().manual_seed(9)
    qkv = torch.randn(L * B, 3 * 64 * H, generator=g) * 0.5
    out = torch.full((L * B, 64 * H), 5.0, device="cuda")
    ql = torch.tensor([300], dtype=torch.int32, device="cuda")
    ops.attention_f32(qkv.cuda(), torch.tensor(lengths, dtype=torch.int32).cuda(), L, B, H, True, out=out,
                      q_limit=ql)
    ref = _attn_ref(qkv, lengths, L, B, H, True)
    got = out.view(L, B, 64 * H).double().cpu()
    for b, n in enumerate(lengths):
        assert _rel(got[:n, b], ref[:n, b]) <= TOL_ATTN
    assert bool((got[384:] == 5.0).all())  # tiles starting at or beyond q_limit are untouched


# ------------------------------------------------------------------------------------- conv front end
@pytest.mark.parametrize("C,T,Fd", [(64, 1001, 40), (128, 333, 80)])
def test_conv_front_end_f32(C, T, Fd):
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(C + T)
    x = torch.randn(2, T, Fd, generator=g)
    w1, b1 = torch.randn(C, 1, 3, 3, generator=g) / 3, torch.randn(C, generator=g) * 0.1
    w2, b2 = torch.randn(C, C, 3, 3, generator=g) / math.sqrt(9 * C), torch.randn(C, generator=g) * 0.1
    s1, h1 = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.1
    s2, h2 = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.1
    y = F.relu(F.conv2d(x.double()[:, None], w1.double(), b1.double(), stride=2, padding=1))
    y = y * s1.double()[:, None, None] + h1.double()[:, None, None]
    y = F.relu(F.conv2d(y, w2.double(), b2.double(), stride=2, padding=1))
    y = y * s2.double()[:, None, None] + h2.double()[:, None, None]
    ref = y.permute(0, 2, 3, 1)  # [B, T2, F2, C]
    c = lambda t: t.cuda()  # noqa: E731
    y1 = ops.conv1_relu_bn_f32(c(x), c(w1.reshape(C, 9)), c(b1), c(s1), c(h1))
    out = ops.conv2_relu_bn_f32(y1, c(ops.prep_conv2_weight_f32(w2)), c(b2), c(s2), c(h2))
    assert out.shape == ref.shape
    assert _rel(out, ref) <= 1e-5


# ------------------------------------------------------------------------------------------ encoder
def _encoder(model, precision="fp32"):
    from fbkst_b200.config import build_encoder
    torch.manual_seed(0)
    enc = build_encoder(dict(model, precision=precision), None, device="cpu")
    bench.randomise_norm_stats(enc, 1)
    return enc.cuda().eval()


def _bump(enc, plan):
    p = plan.cuda()
    return enc.ctc_fc.register_forward_hook(
        lambda m, i, o: o.scatter_add(2, p.unsqueeze(-1), torch.full_like(o[..., :1], bench.CTC_MARGIN)))


def _check(name, out, ref, cols=None):
    B_ref = ref["encoder_out"].shape[1]
    cols = list(range(B_ref)) if cols is None else cols
    nl = ref["src_lengths"].tolist()
    assert out.src_lengths.cpu()[cols].tolist() == nl, name
    L2 = max(nl)
    if ref["encoder_padding_mask"] is not None:
        assert torch.equal(out.encoder_padding_mask.cpu()[cols][:, :L2], ref["encoder_padding_mask"]), name
    rep = parity_report(out.encoder_out[:L2, cols].float().cpu(), ref["encoder_out"], nl)
    assert rep["max_rel"] <= TOL_F32 and rep["elementwise"] <= TOL_F32, (name, rep)
    return rep


def _oracle(enc, model, x, lens, plan, n=None):
    n = len(lens) if n is None else n
    sd = {k: v.detach().float().cpu() for k, v in enc.state_dict().items()}
    xr = torch.zeros(n, x.shape[1], x.shape[2])
    for b in range(n):
        xr[b, : lens[b]] = O.cmvn(x[b, : lens[b]])
    hook = O.bump_hook(plan[:, :n], bench.CTC_MARGIN) if plan is not None else None
    return O.encoder_forward(sd, model, xr, torch.as_tensor(lens[:n]), ctc_logits_hook=hook)


def _run(enc, x, lens):
    from fbkst_b200 import ops
    xn = ops.cmvn(x.cuda(), lens.to(torch.int32).cuda())
    return xn, enc(xn, lens.cuda())


def test_cfg1_full_depth_vs_oracle():
    cfgb = bench.CONFIGS["cfg1"]
    model, lengths = cfgb["model"], cfgb["lengths"]
    B, T = len(lengths), max(lengths)
    L = ((T + 1) // 2 + 1) // 2
    enc = _encoder(model)
    plan = bench.label_plan(L, B, model["vocab"], seed=3)
    _bump(enc, plan)
    x, lens = bench.make_batch(lengths, model["feat_dim"], 1234)
    xn, out = _run(enc, x, lens)
    ref = _oracle(enc, model, x, lengths, plan)
    _check("cfg1/fp32/eager", out, ref)
    # CTC labels exact: the logits of both sides give the same frame arg-max over the valid frames
    sub = [((n + 1) // 2 + 1) // 2 for n in lengths]
    for b, n in enumerate(sub):
        assert torch.equal(out.ctc_out[:n, b].argmax(-1).cpu(), ref["ctc_out"][:n, b].argmax(-1))
    rep = parity_report(out.ctc_out.float().cpu(), ref["ctc_out"], sub)
    assert rep["max_rel"] <= TOL_F32
    enc.use_cuda_graph = True
    out_g = enc(xn, lens)
    assert torch.equal(out_g.encoder_out, out.encoder_out), "graph replay != eager launches"
    assert torch.equal(out_g.src_lengths, out.src_lengths)


@pytest.mark.parametrize("strategy", ["avg", "weighted", "softmax"])
def test_cfg2_vs_oracle(strategy):
    """The bench's cfg2 model at its 11 layers, compression at 8; the oracle computes 4 of 16 utterances."""
    model = dict(bench.CONFIGS["cfg2"]["model"], ctc_strategy=strategy)
    lengths = [1500] * 16
    L = 375
    enc = _encoder(model)
    plan = bench.label_plan(L, len(lengths), model["vocab"], seed=7)
    _bump(enc, plan)
    x, lens = bench.make_batch(lengths, 40, 4321)
    xn, out = _run(enc, x, lens)
    ref = _oracle(enc, model, x, lengths, plan, n=4)
    _check("cfg2/%s/fp32/eager" % strategy, out, ref, cols=[0, 1, 2, 3])
    enc.use_cuda_graph = True
    out_g = enc(xn, lens)
    assert torch.equal(out_g.encoder_out, out.encoder_out)


def test_ragged_odd_lengths_vs_oracle():
    model = dict(bench.CONFIGS["cfg2"]["model"], layers=5, ctc_layer=3, ctc_strategy="weighted")
    lengths = [1601, 1333, 999, 801, 403, 250, 201, 37]
    B, T = len(lengths), max(lengths)
    L = ((T + 1) // 2 + 1) // 2
    enc = _encoder(model)
    plan = bench.label_plan(L, B, model["vocab"], seed=11)
    _bump(enc, plan)
    x, lens = bench.make_batch(lengths, 40, 99)
    xn, out = _run(enc, x, lens)
    ref = _oracle(enc, model, x, lengths, plan)
    _check("ragged/fp32/eager", out, ref)
    enc.use_cuda_graph = True
    out_g = enc(xn, lens.cuda())
    assert torch.equal(out_g.encoder_out, out.encoder_out)


def test_no_penalty_no_compression_vs_oracle():
    model = dict(embed_dim=256, ffn_dim=1024, heads=4, layers=3, conv_channels=128, feat_dim=80, vocab=50,
                 distance_penalty=None, ctc_layer=0)
    lengths = [901, 640, 333]
    enc = _encoder(model)
    x, lens = bench.make_batch(lengths, 80, 5)
    _, out = _run(enc, x, lens)
    ref = _oracle(enc, model, x, lengths, None)
    _check("nopen/fp32/eager", out, ref)


def test_return_all_hiddens():
    model = dict(bench.CONFIGS["cfg1"]["model"])
    lengths = [1000, 777, 501]
    L = 250
    enc = _encoder(model)
    plan = bench.label_plan(L, len(lengths), model["vocab"], seed=2)
    _bump(enc, plan)
    x, lens = bench.make_batch(lengths, 40, 8)
    from fbkst_b200 import ops
    xn = ops.cmvn(x.cuda(), lens.to(torch.int32).cuda())
    out = enc(xn, lens, return_all_hiddens=True)
    plain = enc(xn, lens)
    assert len(out.encoder_states) == model["layers"]
    assert torch.equal(out.src_lengths, plain.src_lengths)
    L2 = int(out.src_lengths.max())
    assert out.encoder_states[-1].shape == (L2, len(lengths), model["embed_dim"])
    assert torch.allclose(out.encoder_out, plain.encoder_out[:L2], rtol=0, atol=1e-5)
    ref = _oracle(enc, model, x, lengths, plan)
    _check("hiddens/fp32", out, ref)


def test_bf16_path_unaffected_by_precision_switch():
    """The default path gives bit-identical outputs before and after the same encoder ran in fp32."""
    model = dict(bench.CONFIGS["cfg1"]["model"])
    lengths = bench.CONFIGS["cfg1"]["lengths"]
    enc = _encoder(model, precision="bf16")
    x, lens = bench.make_batch(lengths, 40, 1234)
    xn = x.cuda()
    before = enc(xn, lens.cuda())
    enc.precision = "fp32"
    f32 = enc(xn, lens.cuda())
    enc.precision = "bf16"
    after = enc(xn, lens.cuda())
    assert torch.equal(before.encoder_out, after.encoder_out) and torch.equal(before.ctc_out, after.ctc_out)
    assert not torch.equal(f32.encoder_out, before.encoder_out) or f32.encoder_out.shape != before.encoder_out.shape
    enc.use_cuda_graph = True
    g_bf16 = enc(xn, lens)
    enc.precision = "fp32"
    g_f32 = enc(xn, lens)
    assert torch.equal(g_bf16.encoder_out, before.encoder_out)
    assert torch.equal(g_f32.encoder_out, f32.encoder_out)


def test_half_model_hands_fp16_to_the_decoder():
    enc = _encoder(dict(bench.CONFIGS["cfg1"]["model"])).half()
    x, lens = bench.make_batch([800, 640], 40, 1)
    out = enc(x.cuda(), lens.cuda())
    assert out.encoder_out.dtype == torch.float16


def test_training_raises():
    enc = _encoder(dict(bench.CONFIGS["cfg1"]["model"]))
    enc.train()
    x, lens = bench.make_batch([400], 40, 1)
    with pytest.raises(NotImplementedError, match="inference only"):
        enc(x.cuda(), lens.cuda())
