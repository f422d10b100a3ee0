"""GPU parity of every kernel, called through the C ABI (fbkst_b200.ops -> ctypes), against the
CPU oracle / golden vectors made from the live reference, or a plain fp32 PyTorch formula.

Tolerances (BASELINE.json north_star): integer outputs bit-exact; bf16-path floats 2e-2
relative to the tensor's max magnitude; fp32 kernels 1e-3 or tighter."""
import math
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import encoder_oracle as O  # noqa: E402  (checker only)


def dev():
    return torch.device("cuda:0")


def rel_err(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-12)).item()


def bf(x):
    return x.to(torch.bfloat16)


# ------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 256, 128), (300, 512, 512), (1000, 1536, 512),
                                   (77, 200, 640), (513, 2048, 512), (640, 512, 2048), (130, 1005, 256)])
def test_linear_plain(M, N, K):
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(M + N + K)
    a = bf(torch.randn(M, K, generator=g)).to(dev())
    w = bf(torch.randn(N, K, generator=g) / math.sqrt(K)).to(dev())
    bias = torch.randn(N, generator=g).to(dev())
    ref = a.float() @ w.float().t() + bias
    out = ops.linear(a, w, bias, out_dtype=torch.float32)
    torch.cuda.synchronize()
    assert out.shape == (M, N)
    e = rel_err(out, ref)
    assert e < 1e-4, (M, N, K, e)
    out = ops.linear(a, w, bias, relu=True)
    e = rel_err(out.float(), torch.relu(ref))
    assert e < 1e-2, (M, N, K, e)


@pytest.mark.parametrize("M,N,K", [(300, 512, 640), (1000, 256, 640), (77, 1024, 2560)])
def test_linear_fp16_operands(M, N, K):
    """fc3's operand pair (conv2's fp16 output x fp16 weight, FBKST_EPI_AB_F16): same kernel, fp16
    instruction descriptor; exact products in fp32 accumulation -> 1e-4 against fp32 on the same operands.
    Values are chosen so that a bf16 interpretation of the bits would be wildly off."""
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(M + N + K + 1)
    a = torch.randn(M, K, generator=g).half().to(dev())
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).half().to(dev())
    bias = torch.randn(N, generator=g).to(dev())
    ref = a.float() @ w.float().t() + bias
    out = ops.linear(a, w, bias, relu=True, out_dtype=torch.float32)
    torch.cuda.synchronize()
    assert rel_err(out, torch.relu(ref)) < 1e-4
    with pytest.raises(ValueError):
        ops.linear(a, w.to(torch.bfloat16), bias)  # mixed operand types are rejected


def test_linear_residual():
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(3)
    B, L, K, N = 3, 50, 640, 256
    a = bf(torch.randn(B * L, K, generator=g)).to(dev())
    w = bf(torch.randn(N, K, generator=g) / math.sqrt(K)).to(dev())
    bias = torch.randn(N, generator=g).to(dev())
    res = torch.randn(B * L, N, generator=g).to(dev())
    ref = a.float() @ w.float().t() + bias
    out = ops.linear(a, w, bias, residual=res, out_dtype=torch.float32)
    assert rel_err(out, ref + res) < 1e-4
    # the sinusoidal position table fc3's output receives (embed_remap_stats adds it: test_embed_remap_stats)
    table = ops.sinusoidal_table(L + 1, N, dev())
    assert rel_err(table, O.sinusoidal_table(L + 1, N)) < 1e-5


# ------------------------------------------------------------------------------- LayerNorm
@pytest.mark.parametrize("D", [128, 256, 512, 1024])
def test_layernorm(D):
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(D)
    x = (torch.randn(333, D, generator=g) * 2 + 0.5).to(dev())
    gamma, beta = torch.randn(D, generator=g).to(dev()), torch.randn(D, generator=g).to(dev())
    ref = torch.nn.functional.layer_norm(x, (D,), gamma, beta, 1e-5)
    assert rel_err(ops.layernorm(x, gamma, beta, out_dtype=torch.float32), ref) < 1e-5
    assert rel_err(ops.layernorm(x, gamma, beta).float(), ref) < 1e-2


# --------------------------------------------------------- LayerNorm folded into the GEMMs
def _slice_stats(x):
    """(mean, M2) per 128-column slice, fp64 -> [M, parts, 2]."""
    M, D = x.shape
    parts = (D + 127) // 128
    out = torch.zeros(M, parts, 2, dtype=torch.float64)
    for p in range(parts):
        sl = x[:, p * 128:(p + 1) * 128].double()
        out[:, p, 0] = sl.mean(1)
        out[:, p, 1] = ((sl - sl.mean(1, keepdim=True)) ** 2).sum(1)
    return out


@pytest.mark.parametrize("M,D", [(333, 128), (1000, 256), (777, 512), (300, 1024), (64, 384)])
def test_row_stats_cast(M, D):
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(D + M)
    x = (torch.randn(M, D, generator=g) * 2 + 3.0).to(dev())
    xb, st = ops.row_stats_cast(x)
    torch.cuda.synchronize()
    assert torch.equal(xb, x.to(torch.bfloat16))
    ref = _slice_stats(x.cpu())
    assert rel_err(st[..., 0], ref[..., 0]) < 1e-5
    assert rel_err(st[..., 1], ref[..., 1]) < 1e-5


@pytest.mark.parametrize("L,B,D,pos", [(37, 5, 128, True), (95, 8, 512, True), (61, 3, 1024, True),
                                       (50, 4, 256, False), (1, 1, 384, True)])
def test_embed_remap_stats(L, B, D, pos):
    """(b,t)-ordered fc3 output -> time-major rows + sinusoidal positions (table row t+1 inside the
    utterance, the padding row beyond it: conv_transformer.py:225-229, positional_embedding_audio.py:20-26)
    + bf16 copy + slice statistics; the fp32 result is bit-exact (one fp32 add per element)."""
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(L * 7 + D)
    src = torch.randn(B * L, D, generator=g).to(dev())
    lengths = torch.randint(1, L + 1, (B,), generator=g).to(torch.int32)
    lengths[0] = L
    table = ops.sinusoidal_table(L + 8, D, dev()) if pos else None
    x, xb, st = ops.embed_remap_stats(src, L, B, table, lengths.to(dev()) if pos else None)
    torch.cuda.synchronize()
    ref = src.view(B, L, D).transpose(0, 1)
    if pos:
        t = torch.arange(L).view(L, 1)
        rows = torch.where(t < lengths.view(1, B).long(), t + 1, torch.zeros_like(t)).to(dev())  # [L, B]
        ref = ref + table[rows]
    ref = ref.reshape(L * B, D).contiguous()
    assert torch.equal(x, ref)
    assert torch.equal(xb, ref.to(torch.bfloat16))
    rs = _slice_stats(ref.cpu())
    assert rel_err(st[..., 0], rs[..., 0]) < 1e-5
    assert rel_err(st[..., 1], rs[..., 1]) < 1e-5


@pytest.mark.parametrize("M,N,K", [(300, 512, 512), (1000, 256, 1024), (513, 512, 2048), (77, 128, 256),
                                   (640, 1024, 512), (130, 192, 64)])
def test_linear_ln_producer(M, N, K):
    """Residual epilogue that also emits bf16(out) and the per-slice row statistics of out."""
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(M + N + K)
    a = bf(torch.randn(M, K, generator=g)).to(dev())
    w = bf(torch.randn(N, K, generator=g) / math.sqrt(K)).to(dev())
    bias = torch.randn(N, generator=g).to(dev())
    res = (torch.randn(M, N, generator=g) * 2 + 1.5).to(dev())
    ref = a.float() @ w.float().t() + bias + res
    out, xb, st = ops.linear_ln(a, w, bias, residual=res, out_dtype=torch.float32, ln_out=True)
    torch.cuda.synchronize()
    assert rel_err(out, ref) < 1e-4
    assert torch.equal(xb, out.to(torch.bfloat16)), "bf16 copy must be the rounding of the fp32 output"
    exp = _slice_stats(out.cpu())
    assert rel_err(st[..., 0], exp[..., 0]) < 1e-5
    assert rel_err(st[..., 1], exp[..., 1]) < 1e-4
    # same fp32 result as the plain residual epilogue, bit for bit
    assert torch.equal(out, ops.linear(a, w, bias, residual=res, out_dtype=torch.float32))


@pytest.mark.parametrize("M,D,N", [(300, 512, 1536), (1000, 256, 768), (513, 1024, 4096), (77, 128, 256),
                                   (200, 384, 1000)])
def test_linear_ln_consumer(M, D, N):
    """LN(x) W^T + b through the folded form: bf16(x), slice statistics, W'' and c."""
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(M + N + D)
    x = (torch.randn(M, D, generator=g) * 1.7 + 0.6 * torch.randn(M, 1, generator=g)).to(dev())
    gamma = (1 + 0.2 * torch.randn(D, generator=g)).to(dev())
    beta = (0.3 * torch.randn(D, generator=g)).to(dev())
    w = (torch.randn(N, D, generator=g) / math.sqrt(D)).to(dev())
    b = torch.randn(N, generator=g).to(dev())
    scale = torch.ones(N, device=dev())
    scale[: N // 3] = 0.125
    ref = (torch.nn.functional.layer_norm(x.double(), (D,), gamma.double(), beta.double(), 1e-5)
           @ w.double().t() + b.double()) * scale.double()
    xb, st = ops.row_stats_cast(x)
    wf, cf = ops.fold_layernorm(w, b, gamma, beta, row_scale=scale)
    out = ops.linear_ln(xb, wf, cf, stats_in=st, ln_eps=1e-5, out_dtype=torch.float32)
    torch.cuda.synchronize()
    assert rel_err(out, ref) < 1e-2, rel_err(out, ref)
    # not worse than the unfused bf16 path (LayerNorm kernel -> bf16 -> GEMM) beyond noise
    h = ops.layernorm(x, gamma, beta)
    unf = ops.linear(h, ops.cast_bf16(w * scale[:, None]), b * scale, out_dtype=torch.float32)
    assert rel_err(out, ref) < 2.0 * rel_err(unf, ref) + 1e-3
    outr = ops.linear_ln(xb, wf, cf, stats_in=st, relu=True)
    assert rel_err(outr.float(), torch.relu(ref)) < 2e-2


def test_linear_ln_chain_rows_limit():
    """producer -> consumer chained on device with a device-side row limit (post-compression mode)."""
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(11)
    M, D, Dff, Bm = 512, 512, 2048, 8
    a = bf(torch.randn(M, Dff, generator=g)).to(dev())
    w2 = bf(torch.randn(D, Dff, generator=g) / math.sqrt(Dff)).to(dev())
    b2 = torch.randn(D, generator=g).to(dev())
    res = torch.randn(M, D, generator=g).to(dev())
    gamma, beta = torch.ones(D, device=dev()), torch.zeros(D, device=dev())
    w = (torch.randn(3 * D, D, generator=g) / math.sqrt(D)).to(dev())
    b = torch.randn(3 * D, generator=g).to(dev())
    wf, cf = ops.fold_layernorm(w, b, gamma, beta)
    limit = torch.tensor([37], dtype=torch.int32, device=dev())  # 37 * 8 = 296 valid rows
    rows = 37 * Bm
    x = torch.zeros(M, D, device=dev())
    xb = torch.zeros(M, D, dtype=torch.bfloat16, device=dev())
    st = torch.zeros(M, D // 128, 2, device=dev())
    ops.linear_ln(a, w2, b2, residual=res, out_dtype=torch.float32, out=x, ln_out=(xb, st),
                  rows_limit=(limit, Bm))
    y = torch.zeros(M, 3 * D, dtype=torch.bfloat16, device=dev())
    ops.linear_ln(xb, wf, cf, stats_in=st, out=y, rows_limit=(limit, Bm))
    torch.cuda.synchronize()
    xr = a[:rows].float() @ w2.float().t() + b2 + res[:rows]
    assert rel_err(x[:rows], xr) < 1e-4
    yr = torch.nn.functional.layer_norm(xr, (D,)) @ w.t() + b
    assert rel_err(y[:rows].float(), yr) < 2e-2
    # warps whose 32-row block starts beyond the limit write nothing: rows >= 320 keep their zeros
    assert float(y[320:].float().abs().max()) == 0.0
    assert float(x[320:].abs().max()) == 0.0


# ------------------------------------------------------------------------------------ CMVN
def test_cmvn_golden(golden_dir):
    from fbkst_b200 import ops
    cases = torch.load(os.path.join(golden_dir, "cmvn.pt"), weights_only=False)
    for c in cases:
        x = c["x"]
        T, Fd = x.shape
        xb = torch.zeros(2, T + 5, Fd)
        xb[0, :T] = x
        xb[1, : T // 2 + 1] = x[: T // 2 + 1]
        lengths = torch.tensor([T, T // 2 + 1], dtype=torch.int32)
        y = ops.cmvn(xb.to(dev()), lengths.to(dev())).cpu()
        assert rel_err(y[0, :T], c["y"]) < 1e-4
        assert y[0, T:].abs().max() == 0 and y[1, T // 2 + 1:].abs().max() == 0
        if T // 2 + 1 >= 2:
            assert rel_err(y[1, : T // 2 + 1], O.cmvn(x[: T // 2 + 1])) < 1e-4


# ----------------------------------------------------------------------------------- convs
def conv_ref(x, w, b, gamma, beta, mean, var):
    y = torch.nn.functional.conv2d(x, w, b, stride=2, padding=1)
    return torch.nn.functional.batch_norm(torch.relu(y), mean, var, gamma, beta, False, 0.0, 1e-5)


@pytest.mark.parametrize("B,T,Fd,C", [(2, 61, 40, 64), (3, 100, 40, 64), (2, 37, 80, 64), (2, 45, 80, 128),
                                      (1, 7, 40, 64), (2, 130, 42, 64)])
def test_conv_stack(B, T, Fd, C):
    """conv1 (tcgen05) then conv2 (TMA implicit GEMM, tcgen05) vs F.conv2d+ReLU+BN (eval)."""
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(B * T + Fd)
    x = torch.randn(B, T, Fd, generator=g)
    w1 = torch.randn(C, 1, 3, 3, generator=g) * 0.6
    w2 = torch.randn(C, C, 3, 3, generator=g) * (1.0 / math.sqrt(9 * C))
    b1, b2 = torch.randn(C, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1
    bn = [(1 + 0.1 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g),
           0.1 * torch.randn(C, generator=g), torch.rand(C, generator=g) + 0.5) for _ in range(2)]
    r1 = conv_ref(x.unsqueeze(1), w1, b1, *bn[0])
    d = dev()
    s0 = ops.prep_bn_affine(*[t.to(d) for t in bn[0]])
    s1 = ops.prep_bn_affine(*[t.to(d) for t in bn[1]])
    y1 = ops.conv1_relu_bn(x.to(d), w1.reshape(C, 9).contiguous().to(d), b1.to(d), *s0)
    assert y1.shape == (B, (T + 1) // 2, (Fd + 1) // 2, C)
    assert y1.dtype == torch.float16  # the conv front end runs in IEEE fp16 (fp32 accumulation)
    e1 = rel_err(y1.float().permute(0, 3, 1, 2), r1)
    assert e1 < 2.5e-3, e1  # fp16 operands: 4x tighter than the former bf16 bound
    # conv2 reference consumes OUR fp16 conv1 output so the test isolates conv2
    r2 = conv_ref(y1.float().permute(0, 3, 1, 2).cpu(), w2.half().float(), b2, *bn[1])
    y2 = ops.conv2_relu_bn(y1, ops.prep_conv2_weight(w2.to(d)), b2.to(d), *s1)
    torch.cuda.synchronize()
    assert y2.shape == (B, r2.shape[2], r2.shape[3], C)
    e2 = rel_err(y2.float().permute(0, 3, 1, 2), r2)
    assert e2 < 2.5e-3, e2


def test_fc3_weight_permutation():
    from fbkst_b200 import ops
    D, C, F2 = 128, 64, 10
    w = torch.randn(D, C * F2)
    p = ops.prep_fc3_weight(w.to(dev()), C, F2).float().cpu()
    exp = w.view(D, C, F2).permute(0, 2, 1).reshape(D, F2 * C).half().float()
    assert torch.equal(p, exp)


# ------------------------------------------------------------------------------- attention
def attn_ref(qkv, lengths, L, B, H, log_penalty):
    """local_attention.py:115-139 in fp32 on (already scaled) q."""
    D = H * 64
    q, k, v = qkv.float().view(L, B, 3, H, 64).permute(2, 1, 3, 0, 4)  # [3] B H L 64
    s = q @ k.transpose(-1, -2)
    key_pad = torch.arange(L, device=qkv.device)[None, :] >= lengths[:, None]
    s = s.masked_fill(key_pad[:, None, None, :], float("-inf"))
    if log_penalty:
        i = torch.arange(L, device=qkv.device)
        s = s - torch.clamp(torch.log((i[:, None] - i[None, :]).abs().float()), min=0)
    o = torch.softmax(s, -1) @ v  # B H L 64
    return o.permute(2, 0, 1, 3).reshape(L * B, D)


@pytest.mark.parametrize("L,B,H,lens,pen", [
    (128, 2, 2, [128, 128], True), (100, 3, 2, [100, 64, 5], True), (375, 2, 8, [375, 201], True),
    (300, 2, 4, [300, 129], False), (700, 1, 2, [700], True),
    (1700, 1, 2, [1700], True), (2100, 2, 1, [2100, 1300], False),  # long inputs on the default kernel (L <~ 2500)
    # more work items than persistent CTAs (several items per CTA, item boundaries inside the
    # flattened key-tile stream), ragged lengths incl. tiles of padded queries
    (375, 24, 8, [375] * 6 + [300] * 6 + [190] * 6 + [64, 65, 127, 128, 129, 1], True),
    (200, 48, 4, [200 - 3 * i for i in range(48)], False)])
def test_attention(L, B, H, lens, pen):
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(L + B)
    qkv = bf(torch.randn(L * B, 3 * H * 64, generator=g) * 0.7).to(dev())
    lengths = torch.tensor(lens, dtype=torch.int32, device=dev())
    out = ops.attention(qkv, lengths, L, B, H, pen).float().view(L, B, H * 64)
    torch.cuda.synchronize()
    ref = attn_ref(qkv, lengths, L, B, H, pen).view(L, B, H * 64)
    for b, n in enumerate(lens):  # only valid query rows are defined by the reference
        e = rel_err(out[:n, b], ref[:n, b])
        assert e < 2e-2, (b, n, e)
    assert torch.isfinite(out).all()


@pytest.mark.parametrize("pattern", ["ramp", "late_spike", "second_half", "second_tile_128"])
@pytest.mark.parametrize("pen", [True, False])
def test_attention_growing_scores(pattern, pen):
    """The one-pass softmax takes its running reference from the first 32 columns of the first key tile and raises it
    only when a later half-tile exceeds it by 2^24: scores that GROW along the key axis drive both rare paths (the
    first-half raise with the rescale of O / l, and the restart of a tile whose second half overflows)."""
    from fbkst_b200 import ops
    L, B, H = 375, 2, 2
    lens = [375, 230]
    g = torch.Generator().manual_seed(11)
    qkv = torch.randn(L, B, 3, H, 64, generator=g) * 0.3
    u = torch.randn(64, generator=g)
    u = u / u.norm()
    j = torch.arange(L, dtype=torch.float32)
    if pattern == "ramp":            # +0.75 nats per key: every 32-column half is 24 nats above the previous one
        amp = 0.75 * j
    elif pattern == "late_spike":    # flat, then a few keys 60-90 nats above everything seen so far
        amp = torch.zeros(L)
        amp[150] = 60.0
        amp[151] = 59.0
        amp[300] = 150.0
    elif pattern == "second_tile_128":  # keys 198..237 of the second 128-key tile jump (raise + rescale of O / l
        amp = torch.zeros(L)            # in the wide kernel, whose tiles are 128 keys)
        amp[128 + 70: 128 + 110] = 45.0
    else:                            # only the SECOND half of the third tile jumps (restart path, no earlier hint)
        amp = torch.zeros(L)
        amp[64 * 2 + 40: 64 * 2 + 64] = 45.0
    qkv[:, :, 0] = qkv[:, :, 0] * 0.1 + u          # q ~ u (norm ~1)
    qkv[:, :, 1] = qkv[:, :, 1] * 0.1 + amp[:, None, None, None] * u
    qkv = bf(qkv.reshape(L * B, 3 * H * 64)).to(dev())
    lengths = torch.tensor(lens, dtype=torch.int32, device=dev())
    out = ops.attention(qkv, lengths, L, B, H, pen).float().view(L, B, H * 64)
    torch.cuda.synchronize()
    ref = attn_ref(qkv, lengths, L, B, H, pen).view(L, B, H * 64)
    assert torch.isfinite(out).all()
    for b, n in enumerate(lens):
        e = rel_err(out[:n, b], ref[:n, b])
        assert e < 2e-2, (pattern, b, n, e)


# ------------------------------------------------------------------------------------- CTC
def run_ctc(x, logits, lengths, strategy):
    from fbkst_b200 import ops
    L, B, V = logits.shape
    D = x.shape[-1]
    d = dev()
    lg = logits.to(d).reshape(L * B, V)
    ln = lengths.to(torch.int32).to(d)
    labels, prob = ops.ctc_argmax(lg, ln, L, B, V, want_prob=strategy != "avg")
    seg_id, seg_start, weight, new_len, max_new = ops.ctc_segment(labels, prob, ln, strategy, L, B)
    out = ops.ctc_compress(x.to(d).reshape(L * B, D).contiguous(), seg_id, seg_start, weight, ln, new_len,
                           max_new, L, B)
    nl = new_len.cpu()
    L2 = int(max_new.item())
    return out[: L2 * B].view(L2, B, D).cpu(), nl.long(), labels.view(L, B).cpu(), seg_id.view(L, B).cpu()


def test_ctc_compress_golden(golden_dir):
    cases = torch.load(os.path.join(golden_dir, "ctc_compress.pt"), weights_only=False)
    for c in cases:
        out, nl, labels, seg_id = run_ctc(c["x"], c["logits"], c["lengths"], c["strategy"])
        assert torch.equal(nl, c["new_lengths"].long()), c["name"]
        segs = O.ctc_segments(c["logits"], c["lengths"])
        for b, sg in enumerate(segs):  # labels and segment boundaries bit-exact
            exp_lab = [lab for lab, run in sg for _ in range(run)]
            exp_seg = [s for s, (lab, run) in enumerate(sg) for _ in range(run)]
            n = int(c["lengths"][b])
            assert labels[:n, b].tolist() == exp_lab, c["name"]
            assert seg_id[:n, b].tolist() == exp_seg, c["name"]
            assert (labels[n:, b] == -1).all() and (seg_id[n:, b] == -1).all()
        assert out.shape == c["out"].shape, c["name"]
        assert rel_err(out, c["out"]) < 1e-5, c["name"]


def test_ctc_argmax_bf16_unaligned_and_ties():
    """bf16 logits with an odd V (rows not 16-byte aligned) and exact ties -> lowest index."""
    from fbkst_b200 import ops
    L, B, V = 9, 3, 1005
    g = torch.Generator().manual_seed(0)
    logits = bf(torch.randn(L, B, V, generator=g))
    logits[0, 0, 17] = logits[0, 0, 900] = 9.0      # tie -> 17
    logits[1, 1, 1004] = 11.0                       # last column
    logits[2, 2, 0] = 12.0                          # first column
    lengths = torch.tensor([9, 9, 4], dtype=torch.int32)
    labels, prob = ops.ctc_argmax(logits.to(dev()).view(L * B, V), lengths.to(dev()), L, B, V)
    labels = labels.view(L, B).cpu()
    ref = logits.float().argmax(-1)
    for b in range(B):
        n = int(lengths[b])
        assert labels[:n, b].tolist() == ref[:n, b].tolist()
        assert (labels[n:, b] == -1).all()
    assert labels[0, 0] == 17 and labels[1, 1] == 1004 and labels[2, 2] == 0
    p_ref = torch.softmax(logits.float(), -1).max(-1).values
    p = prob.view(L, B).cpu()
    assert rel_err(p[:4], p_ref[:4]) < 1e-4


def test_ctc_full_size_properties():
    """cfg2-sized compression (L=375, B=64, V=8005): size-independent properties --
    new lengths == number of label changes, every column of W sums to 1 (out of a constant
    input is that constant), padding rows are exactly 0."""
    from fbkst_b200 import ops
    L, B, V, D = 375, 64, 8005, 512
    d = dev()
    labels_plan = O.synthetic_ctc_bump(L, B, V, seed=3)
    g = torch.Generator().manual_seed(1)
    lens = torch.randint(200, L + 1, (B,), generator=g).sort(descending=True).values
    lens[0] = L
    logits = torch.randn(L, B, V, generator=g, dtype=torch.float32).bfloat16()
    logits = O.bump_hook(labels_plan, 8.0)(logits.float()).bfloat16()
    x = torch.ones(L * B, D, device=d) * 1.5
    ln = lens.to(torch.int32).to(d)
    for strategy in ("avg", "weighted", "softmax"):
        lab, prob = ops.ctc_argmax(logits.to(d).view(L * B, V), ln, L, B, V, want_prob=strategy != "avg")
        seg_id, seg_start, weight, new_len, max_new = ops.ctc_segment(lab, prob, ln, strategy, L, B)
        out = ops.ctc_compress(x, seg_id, seg_start, weight, ln, new_len, max_new, L, B)
        lab = lab.view(L, B).cpu()
        nl = new_len.cpu()
        L2 = int(max_new.item())
        out = out[: L2 * B].view(L2, B, D).cpu()
        for b in range(0, B, 7):
            n = int(lens[b])
            assert lab[:n, b].tolist() == labels_plan[:n, b].tolist()
            changes = 1 + int((lab[1:n, b] != lab[: n - 1, b]).sum())
            assert int(nl[b]) == changes
            assert torch.allclose(out[: changes, b], torch.full((changes, D), 1.5), atol=1e-5)
            assert out[changes:, b].abs().max() == 0
        assert L2 == int(nl.max())


def test_torch_custom_ops_match_direct_calls():
    """torch.ops.fbkst.* end in the same extern "C" entry points as fbkst_b200.ops.*."""
    from fbkst_b200 import ops, torch_ops  # noqa: F401
    g = torch.Generator().manual_seed(0)
    a = bf(torch.randn(300, 256, generator=g)).to(dev())
    w = bf(torch.randn(384, 256, generator=g) * 0.05).to(dev())
    bias = torch.randn(384, generator=g).to(dev())
    res = torch.randn(300, 384, generator=g).to(dev())
    assert torch.equal(torch.ops.fbkst.linear(a, w, bias, True, None, False), ops.linear(a, w, bias, relu=True))
    assert torch.equal(torch.ops.fbkst.linear(a, w, bias, False, res, True),
                       ops.linear(a, w, bias, residual=res, out_dtype=torch.float32))
    x = torch.randn(300, 256, generator=g).to(dev())
    gm, bt = torch.randn(256, generator=g).to(dev()), torch.randn(256, generator=g).to(dev())
    assert torch.equal(torch.ops.fbkst.layernorm(x, gm, bt, False, 1e-5), ops.layernorm(x, gm, bt))
    L, B, H = 100, 3, 2
    qkv = bf(torch.randn(L * B, 3 * H * 64, generator=g) * 0.7).to(dev())
    lens = torch.tensor([100, 64, 5], dtype=torch.int32, device=dev())
    assert torch.equal(torch.ops.fbkst.attention(qkv, lens, L, B, H, True), ops.attention(qkv, lens, L, B, H, True))
    V, D = 50, 128
    logits = torch.randn(L * B, V, generator=g).to(dev())
    xs = torch.randn(L * B, D, generator=g).to(dev())
    lab, prob = torch.ops.fbkst.ctc_argmax(logits, lens, L, B, V, True)
    seg_id, seg_start, weight, new_len, max_new = torch.ops.fbkst.ctc_segment(lab, prob, lens, "weighted", L, B)
    out = torch.ops.fbkst.ctc_compress(xs, seg_id, seg_start, weight, lens, new_len, max_new, L, B)
    lab2, prob2 = ops.ctc_argmax(logits, lens, L, B, V, True)
    s2 = ops.ctc_segment(lab2, prob2, lens, "weighted", L, B)
    out2 = ops.ctc_compress(xs, s2[0], s2[1], s2[2], lens, s2[3], s2[4], L, B)
    n = int(max_new.item()) * B
    assert torch.equal(lab, lab2) and torch.equal(new_len, s2[3]) and torch.equal(out[:n], out2[:n])
    mask = torch.ops.fbkst.lengths_to_mask(lens, L)
    assert mask.dtype == torch.bool and mask.shape == (B, L) and bool(mask[2, 5]) and not bool(mask[2, 4])


# ------------------------------------------------------------------ next row N2: device collater
def test_device_collater_reference_kat():
    """The reference's collate KAT (tests/speech_recognition/test_collaters.py:23-50) through the
    device collater: same ids / lengths / targets, src_tokens padded on the device."""
    import numpy as np
    from fbkst_b200.data import DeviceCollater
    s1 = {"id": 0, "data": [np.array([[7, 8], [9, 10]]), np.array([4, 2, 3, 1])]}
    s2 = {"id": 1, "data": [np.array([[1, 2], [3, 4], [5, 6]]), np.array([3, 2, 1])]}
    batch = DeviceCollater(0, 1, pad_index=0, eos_index=1).collate([s1, s2])
    assert batch["id"].tolist() == [1, 0] and batch["ntokens"] == 7 and batch["nsentences"] == 2
    assert batch["net_input"]["src_tokens"].is_cuda
    assert batch["net_input"]["src_tokens"].cpu().tolist() == [[[1, 2], [3, 4], [5, 6]], [[7, 8], [9, 10], [0, 0]]]
    assert batch["net_input"]["prev_output_tokens"].tolist() == [[1, 3, 2, 0], [1, 4, 2, 3]]
    assert batch["net_input"]["src_lengths"].tolist() == [3, 2]
    assert batch["target"].tolist() == [[3, 2, 1, 0], [4, 2, 3, 1]]


@pytest.mark.parametrize("normalize", [False, True])
def test_device_collater_vs_oracle(normalize):
    """Ragged utterances -> padded (and normalised) batch: bit-exact copy without CMVN, 1e-5 with."""
    from oracle import collate_oracle as C
    from fbkst_b200.data import DeviceCollater
    g = torch.Generator().manual_seed(11)
    lens = [1500, 3, 977, 1201, 640, 1, 1500, 333]
    samples = [{"id": i, "data": [(torch.randn(n, 40, generator=g) * 3 + 1).numpy(),
                                  torch.randint(3, 90, (4 + i,), generator=g).numpy()]}
               for i, n in enumerate(lens)]
    if normalize:  # unbiased variance of a single frame is undefined (NaN in the reference too)
        samples = [s for s in samples if s["data"][0].shape[0] > 1]
    ref = C.collate(samples, normalize=normalize)
    col = DeviceCollater(0, 1, normalize=normalize)
    for _ in range(2):  # second call reuses the pinned buffer
        got = col.collate(samples)
    assert got["net_input"]["src_lengths"].tolist() == ref["net_input"]["src_lengths"].tolist()
    assert sorted(got["id"].tolist()) == sorted(ref["id"].tolist())
    x = got["net_input"]["src_tokens"].cpu()
    for k, i in enumerate(ref["id"].tolist()):
        j = got["id"].tolist().index(i)
        a, r = x[j], ref["net_input"]["src_tokens"][k]
        if normalize:
            assert rel_err(a, r) < 1e-5
        else:
            assert torch.equal(a, r)
        assert torch.equal(got["target"][j], ref["target"][k])
        assert torch.equal(got["net_input"]["prev_output_tokens"][j], ref["net_input"]["prev_output_tokens"][k])


# ------------------------------------------------------------- ctc_fc with the fused arg-max epilogue
@pytest.mark.parametrize("L,B,V,K,want_prob", [(50, 3, 105, 256, True), (120, 4, 1005, 512, True),
                                                (64, 5, 8005, 512, False), (33, 2, 8005, 512, True)])
def test_linear_argmax_fused_epilogue(L, B, V, K, want_prob):
    """logits identical to the plain fp32-output GEMM; labels = arg-max of THOSE logits (bit-exact, lowest
    index on ties), top probability / log-sum-exp within 1e-4; the built-in bump equals a scatter-add hook."""
    from fbkst_b200 import ops
    g = torch.Generator().manual_seed(L + V)
    a = bf(torch.randn(L * B, K, generator=g)).to(dev())
    w = bf(torch.randn(V, K, generator=g) / math.sqrt(K)).to(dev())
    bias = torch.randn(V, generator=g).to(dev())
    lens = torch.tensor([L] + [max(1, L - 7 * b) for b in range(1, B)], dtype=torch.int32, device=dev())
    plain = ops.linear(a, w, bias, out_dtype=torch.float32)
    lg, labels, prob, lse = ops.linear_argmax(a, w, bias, lens, L, B, want_prob=want_prob, want_lse=True)
    assert torch.equal(lg, plain)
    valid = (torch.arange(L, device=dev())[:, None] < lens[None, :]).reshape(-1)
    ref_lab = lg.argmax(-1).to(torch.int32)
    assert torch.equal(labels[valid], ref_lab[valid]) and (labels[~valid] == -1).all()
    ref_lse = torch.logsumexp(lg.double(), -1).float()
    assert (lse[valid] - ref_lse[valid]).abs().max() < 1e-3
    if want_prob:
        ref_p = torch.softmax(lg.double(), -1).max(-1).values.float()
        assert ((prob[valid] - ref_p[valid]).abs() / ref_p[valid]).max() < 1e-3
    # the lean epilogue (maxima only; the merge kernel recovers the column from the winning chunk)
    lg3, lab3, _, _ = ops.linear_argmax(a, w, bias, lens, L, B, want_prob=False)
    assert torch.equal(lg3, plain)
    assert torch.equal(lab3[valid], ref_lab[valid]) and (lab3[~valid] == -1).all()
    # ties -> lowest index: duplicate the winning weight row under a lower AND a higher index, in the same
    # 128-column chunk and in other chunks
    top = int(ref_lab[0])
    for lo, hi in (((top - 3) % V, (top + 5) % V), ((top - 131) % V, (top + 259) % V)):
        w2 = w.clone()
        bias2 = bias.clone()
        for j in (lo, hi):
            w2[j] = w2[top]
            bias2[j] = bias2[top]
        for wp in (False, True):
            _, lab2, _, _ = ops.linear_argmax(a, w2, bias2, lens, L, B, want_prob=wp)
            assert int(lab2[0]) == min(top, lo, hi)
    # built-in bump == hook semantics
    plan = torch.randint(0, V, (L * B,), generator=g).to(torch.int32).to(dev())
    lgb, labb, _, _ = ops.linear_argmax(a, w, bias, lens, L, B, want_prob=False, bump=(plan, 30.0))
    hooked = plain.clone()
    hooked.scatter_add_(1, plan.long().unsqueeze(-1), torch.full((L * B, 1), 30.0, device=dev()))
    assert torch.allclose(lgb, hooked, atol=1e-5)
    assert torch.equal(labb[valid], plan[valid])
