"""Self-attention at its length, tile and dispatch limits, against fp64 on the same operands.

``ops.attention`` (bf16) picks its kernel by shape alone (``attention_entry``, csrc/attention_tcgen05.cu):
the wide kernel (attention_wide.cu, 128-key tiles) whenever its shared memory fits -- always without the
penalty, L <= 2560 with it, where the penalty LUT fills shared memory -- and otherwise the split-KV kernel
``attention_fwd_kernel`` (64-key tiles) up to L = 17216; beyond that the call is refused.  The cases below sit
on the edges where such kernels go wrong: lengths at tile multiples +-1, tiles made only of padding, odd work-item
counts (an idle softmax group in the wide kernel), more than the 64 work items per CTA that both kernels keep
decoded in shared memory, the first L of each kernel, the largest L each accepts, and more than 255 key tiles per
query tile (L > 16320 on split-KV, L > 32640 on the wide kernel).  ``ops.attention_f32`` and the two
cross-attention kernels are checked at their own edges.

The reference is fp64 attention on the kernel's own operands for a sample of query rows (the first and last valid
row of every query tile plus random rows), so L = 33000 stays cheap on the host.  ``test_reference_sees_mistakes``
(no GPU) shows that the bound can see the mistakes a kernel makes at these edges."""
import pytest
import torch

Q_SCALE = 0.375         # pre-scaled q: scores of std 3, so that the penalty and the mask change the result
TOL_BF16 = 8e-3         # max-normalised per utterance: bf16 output rounding (2^-8) plus the bf16 P
TOL_F32 = 3e-5          # ops.attention_f32 against fp64 up to a few thousand keys (TOL_ATTN of test_gpu_fp32.py)
# beyond that the error grows with the number of keys the fp32 softmax sums over: measured 7.0e-5 at L = 16500 and
# 1.2e-4 at L = 33000 on a B200 (the same before and after the key-tile count fix), 8x inside the encoder's 1e-3
TOL_F32_LONG = 2e-4
TOL_XATTN = (8e-3, 1e-5)       # bf16 cross-attention: output, weights (test_gpu_xattn.py)
TOL_XATTN_F32 = (1e-5, 1e-6)   # fp32 cross-attention (test_gpu_xattn_fp32.py)

# ---------------------------------------------------------------------------------- host-side restatement
# Shared memory of the inference kernels as the launch code computes it (attention_wide.cu: aw_smem_bytes;
# attention_tcgen05.cu: attention_smem_bytes; cross_attention.cu: xattn_smem_bytes).
SMEM_MAX = 227 * 1024       # per CTA
SMEM_SM = 228 * 1024        # per SM (1 KB of it reserved per resident CTA)
AW_SMEM_FIXED = 2 * 16384 + 3 * 16384 + 2 * 16384 + 2 * 16384 + 256 + 64 * 16 + 1024
AT_SMEM_FIXED = 16384 + 3 * 8192 + 2 * 8192 + 2 * 16384 + 256 + 2 * 2 * 128 * 4 + 64 * 16 + 1024
ITEM_TABLE = 64             # AW_TABLE / AT_TABLE: work items per CTA decoded once into shared memory


def _ceil(a, b):
    return -(-a // b)


def wide_smem(L, pen):
    return AW_SMEM_FIXED + (4 * (4 * 2 * 128 * _ceil(L, 128) + 32) if pen else 0)


def split_smem(L, pen):
    return AT_SMEM_FIXED + (4 * (128 * _ceil(L, 128) + 64 * _ceil(L, 64)) if pen else 0)


def dispatch(L, B, H, pen, sms):
    """(kernel, grid) that attention_entry launches, or (None, 0) when it refuses the shape."""
    n_items = _ceil(L, 128) * B * H
    if wide_smem(L, pen) <= SMEM_MAX:
        return "attention_fwd_wide_kernel", sms if 2 * sms <= n_items else (n_items + 1) // 2
    smem = split_smem(L, pen)
    if smem > SMEM_MAX:
        return None, 0
    per_sm = 2 if 2 * (smem + 1024) <= SMEM_SM else 1
    return "attention_fwd_kernel", min(per_sm * sms, n_items)


def xattn_smem(S):
    return 4 * (1024 + 4) + 4 * (8 * 64 + 8 * 8 * 64 + 8) + 4 * S * 8


XATTN_S_MAX = max(S for S in range(1, 8192) if xattn_smem(S) <= 200 * 1024)


def test_dispatch_limits():
    """The dispatch table the GPU cases below are built on."""
    largest = lambda pred: max(L for L in range(1, 40000) if pred(L))  # noqa: E731
    assert largest(lambda L: wide_smem(L, True) <= SMEM_MAX) == 2560
    assert wide_smem(10 ** 6, False) <= SMEM_MAX  # no penalty: no LUT, any L
    assert largest(lambda L: split_smem(L, True) <= SMEM_MAX) == 17216
    for L, kernel in [(2560, "attention_fwd_wide_kernel"), (2561, "attention_fwd_kernel"),
                      (17216, "attention_fwd_kernel"), (17217, None)]:
        assert dispatch(L, 1, 1, True, 148)[0] == kernel
    assert dispatch(2561, 64, 16, True, 148)[1] == 2 * 148  # two split-KV CTAs per SM at L = 2561
    assert dispatch(32768, 1, 1, False, 148)[0] == "attention_fwd_wide_kernel"
    # more than 255 key tiles of one query tile, inside the accepted range of each kernel
    assert _ceil(16321, 64) == 256 and _ceil(32641, 128) == 256
    assert XATTN_S_MAX == 5694


# ------------------------------------------------------------------------------------------ inputs, reference
def make_qkv(L, B, H, seed, dtype=torch.bfloat16, device="cpu"):
    """[L*B, 3*H*64] (row t*B + b), q pre-scaled by Q_SCALE."""
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.randn(L * B, 3 * H * 64, generator=g, device=device)
    x[:, : 64 * H] *= Q_SCALE
    return x.to(dtype)


def sample_rows(n, seed, extra=8):
    """First and last valid row of every 128-row query tile of an utterance of length n, plus random rows."""
    rows = {r for q0 in range(0, n, 128) for r in (q0, min(q0 + 127, n - 1))}
    rows.update(torch.randint(0, n, (extra,), generator=torch.Generator().manual_seed(seed)).tolist())
    return torch.tensor(sorted(rows))


def log_penalty(d):
    return torch.log(d).clamp_min(0)  # ln(max(1, |i-j|)), 0 on the diagonal


def attn_ref(q, k, v, rows, n_keys, pen, penalty=log_penalty):
    """fp64 attention of query rows ``rows`` (q [R, H, 64]) over keys 0 .. n_keys-1 (k, v [>= n_keys, H, 64])."""
    q, k, v = q.double(), k[:n_keys].double(), v[:n_keys].double()
    out = torch.empty_like(q)
    for c in range(0, len(rows), 256):  # bounded score block at L = 33000
        s = torch.einsum("rhd,jhd->hrj", q[c:c + 256], k)
        if pen:
            d = (rows[c:c + 256, None] - torch.arange(n_keys)[None, :]).abs().double()
            s = s - penalty(d)
        out[c:c + 256] = torch.einsum("hrj,jhd->rhd", torch.softmax(s, -1), v)
    return out


def utterance_operands(qkv, L, B, H, b, rows, n_keys):
    """q at ``rows`` and the first n_keys keys / values of utterance b, on the host."""
    x = qkv.view(L, B, 3, H, 64)
    q = x[rows.to(qkv.device), b, 0].cpu()
    kv = x[:n_keys, b, 1:].cpu()
    return q, kv[:, 0], kv[:, 1]


def max_norm_err(a, ref):
    a, ref = a.double(), ref.double()
    if not bool(torch.isfinite(a).all()):
        return float("inf")
    return ((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


# -------------------------------------------------------------------------------------------- the cases
def _ragged(L):
    """Lengths for a batch of max length L: 1, L, L-1, multiples of 64 and 128 +-1 below L, and (for L > 128)
    utterances whose later query tiles are padding only."""
    lens = {1, L, max(L - 1, 1)}
    for m in (64, 128, 256):
        lens.update(x for x in (m - 1, m, m + 1) if x <= L)
    return sorted(lens, reverse=True)


def _cases():
    """(id, L, B, H, lens, pen, where the inputs are generated); B may be a function of the SM count."""
    cases = []
    for i, L in enumerate([1, 2, 63, 64, 65, 127, 128, 129, 255, 257]):
        for H in (1, 3, 16):
            pen = (i + H) % 2 == 0
            lens = _ragged(L)
            cases.append(("L%d_H%d_%s" % (L, H, "pen" if pen else "nopen"), L, len(lens), H, lens, pen, "cpu"))
    cases += [
        # n_items = 1, and cfg5's 16 heads
        ("one_item", 100, 1, 1, [100], True, "cpu"),
        ("H16_L375", 375, 3, 16, [375, 256, 1], True, "cpu"),
        # the wide kernel at its largest penalty LUT, and the first L on split-KV
        ("wide_max_lut", 2560, 5, 3, [2560, 2433, 1281, 129, 1], True, "cpu"),
        ("split_first", 2561, 5, 3, [2561, 2560, 2497, 128, 1], True, "cpu"),
        ("split_odd_items", 2561, 15, 1, [2561 - 171 * i for i in range(15)], True, "cpu"),
        # n_items = 2 * SMs - 1 / 2 * SMs + 1 on the wide kernel (an idle softmax group / a third item in a CTA)
        ("items_2sm-1", 128, lambda sms: 2 * sms - 1, 1, lambda B: [1 + (b * 37) % 128 for b in range(B)], False,
         "cpu"),
        ("items_2sm+1", 128, lambda sms: 2 * sms + 1, 1, lambda B: [1 + (b * 37) % 128 for b in range(B)], True,
         "cpu"),
        # more than ITEM_TABLE items per CTA (the later ones decoded on the fly), mostly short lengths
        ("over64_wide", 200, lambda sms: _ceil(70 * sms, 2 * 16), 16,
         lambda B: [[1, 5, 64, 65, 127, 128, 129, 200, 17, 3][b % 10] for b in range(B)], True, "cuda"),
        ("over64_split", 2561, lambda sms: _ceil(70 * 2 * sms, 21 * 16), 16,
         lambda B: [[1, 64, 65, 129, 300, 2, 1000, 17][b % 8] if b % 16 else 2561 - b for b in range(B)], True,
         "cuda"),
        # 256 and more key tiles of 64 keys (split-KV) and of 128 keys (wide kernel, no penalty)
        ("ovf_split_16384", 16384, 5, 1, [16384, 16321, 16320, 8193, 1], True, "cpu"),
        ("ovf_split_17216", 17216, 4, 2, [17216, 16385, 16449, 16320], True, "cpu"),
        ("ovf_wide_32768", 32768, 1, 1, [32768], False, "cpu"),
        ("ovf_wide_32700", 32700, 1, 1, [32700], False, "cpu"),
        ("ovf_wide_33000", 33000, 2, 1, [33000, 32641], False, "cpu"),
    ]
    return cases


CASES = _cases()


def resolve(case, sms=None):
    name, L, B, H, lens, pen, where = case
    if callable(B):
        B = B(sms)
    if callable(lens):
        lens = lens(B)
    assert len(lens) == B and max(lens) <= L
    return name, L, B, H, lens, pen, where


def check_against_ref(out, qkv, L, B, H, lens, pen, seed):
    """Worst max-normalised error over the utterances (sampled rows, all heads) against fp64."""
    o = out.view(L, B, H, 64)
    tol = TOL_BF16 if out.dtype == torch.bfloat16 else (TOL_F32 if L <= 4096 else TOL_F32_LONG)
    worst = 0.0
    for b, n in enumerate(lens):
        rows = sample_rows(n, seed + b)
        q, k, v = utterance_operands(qkv, L, B, H, b, rows, n)
        ref = attn_ref(q, k, v, rows, n, pen)
        e = max_norm_err(o[rows.to(o.device), b].cpu(), ref)
        assert e <= tol, (b, n, e)
        worst = max(worst, e)
    return worst


def padded_tiles(L, B, lens, device):
    """[L, B] bool: rows of query tiles that lie wholly beyond the utterance's length."""
    start = torch.tensor([_ceil(n, 128) * 128 for n in lens], device=device)
    return torch.arange(L, device=device)[:, None] >= start[None, :]


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# --------------------------------------------------------------------------------------- bf16, default dispatch
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_attention_bf16_vs_fp64(case):
    from fbkst_b200 import ops
    sms = _sms()
    name, L, B, H, lens, pen, where = resolve(case, sms)
    kernel, grid = dispatch(L, B, H, pen, sms)
    n_items = _ceil(L, 128) * B * H
    if name.startswith("over64"):  # the premise of the case: CTAs that decode items past the table
        assert n_items > ITEM_TABLE * grid, (n_items, grid)
    seed = L * 31 + B * 7 + H
    qkv = make_qkv(L, B, H, seed, device=where).cuda()
    lengths = torch.tensor(lens, dtype=torch.int32, device="cuda")
    out = ops.attention(qkv, lengths, L, B, H, pen)
    again = ops.attention(qkv, lengths, L, B, H, pen)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(out).all())
    assert torch.equal(out, again), "two identical calls differ"
    o = out.view(L, B, H * 64)
    assert bool((o[padded_tiles(L, B, lens, o.device)] == 0).all()), "padded query tiles are not zero"
    worst = check_against_ref(out, qkv, L, B, H, lens, pen, seed)
    print("\n%s: %s grid %d, %d items (%.1f per CTA), max err %.3g" %
          (name, kernel, grid, n_items, n_items / grid, worst))


@pytest.mark.gpu
@pytest.mark.parametrize("L,pen,kernel", [(2560, True, "attention_fwd_wide_kernel<1>"),
                                          (2561, True, "attention_fwd_kernel"),
                                          (17216, True, "attention_fwd_kernel"),
                                          (40000, False, "attention_fwd_wide_kernel<0>")])
def test_attention_dispatch(L, pen, kernel):
    """The kernel each side of a dispatch limit actually runs; past the last one the call is refused."""
    from torch.profiler import ProfilerActivity, profile

    from fbkst_b200 import ops
    qkv = make_qkv(L, 1, 1, 1, device="cuda")
    lengths = torch.tensor([L], dtype=torch.int32, device="cuda")
    ops.attention(qkv, lengths, L, 1, 1, pen)  # module load outside the profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ops.attention(qkv, lengths, L, 1, 1, pen)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events() if "attention_fwd" in e.name}
    assert len(names) == 1 and kernel in names.pop(), names
    assert dispatch(L, 1, 1, pen, _sms())[0] == kernel.split("<")[0]


@pytest.mark.gpu
def test_attention_refuses_past_the_split_kv_limit():
    from fbkst_b200 import ops
    L = 17217
    qkv = torch.zeros(L, 3 * 64, dtype=torch.bfloat16, device="cuda")
    lengths = torch.tensor([L], dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError, match="shared memory"):
        ops.attention(qkv, lengths, L, 1, 1, True)


@pytest.mark.gpu
@pytest.mark.parametrize("L,lens,H", [(500, [375, 1, 129, 200, 128], 3),           # wide kernel
                                      (2561, [2000, 1, 129, 700], 2)])             # split-KV
@pytest.mark.parametrize("limit", [1, 128, 129, "max"])
def test_attention_q_limit(L, lens, H, limit):
    """fbkst_attention_fwd_limited: valid rows as without the limit (bit for bit); tiles wholly beyond the length
    are zero when they start below q_limit and untouched from q_limit on."""
    from fbkst_b200 import ops
    B = len(lens)
    limit = max(lens) if limit == "max" else limit
    qkv = make_qkv(L, B, H, 5 + L).cuda()
    lengths = torch.tensor(lens, dtype=torch.int32, device="cuda")
    full = ops.attention(qkv, lengths, L, B, H, True).view(L, B, H * 64)
    out = torch.full((L * B, H * 64), -3.5, dtype=torch.bfloat16, device="cuda")
    ops.attention(qkv, lengths, L, B, H, True, out=out,
                  q_limit=torch.tensor([limit], dtype=torch.int32, device="cuda"))
    torch.cuda.synchronize()
    o = out.view(L, B, H * 64)
    for b, n in enumerate(lens):
        assert torch.equal(o[:n, b], full[:n, b]), (b, n)
        for q0 in range(_ceil(n, 128) * 128, L, 128):
            want = 0.0 if q0 < limit else -3.5
            assert bool((o[q0:q0 + 128, b] == want).all()), (b, n, q0, limit)


# ---------------------------------------------------------------------------------------------------- fp32
F32_CASES = [("L%d_H%d_%s" % (L, H, "pen" if pen else "nopen"), L, H, _ragged(L), pen)
             for L in (1, 2, 63, 64, 65, 129) for H in (1, 3, 16) for pen in (True, False)]
F32_CASES += [("long_16500_pen", 16500, 1, [16500, 16321], True), ("long_33000_nopen", 33000, 1, [33000], False)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", F32_CASES, ids=[c[0] for c in F32_CASES])
def test_attention_f32_vs_fp64(case):
    from fbkst_b200 import ops
    name, L, H, lens, pen = case
    B = len(lens)
    seed = L * 31 + B * 7 + H
    qkv = make_qkv(L, B, H, seed, dtype=torch.float32).cuda()
    out = ops.attention_f32(qkv, torch.tensor(lens, dtype=torch.int32, device="cuda"), L, B, H, pen)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(out).all())
    o = out.view(L, B, H * 64)
    assert bool((o[padded_tiles(L, B, lens, o.device)] == 0).all())
    worst = check_against_ref(out, qkv, L, B, H, lens, pen, seed)
    print("\nf32 %s: max err %.3g" % (name, worst))


@pytest.mark.gpu
@pytest.mark.parametrize("limit", [1, 129])
def test_attention_f32_q_limit(limit):
    """Tiles starting at or beyond q_limit are untouched; below it, rows are as without the limit."""
    from fbkst_b200 import ops
    L, H, lens = 300, 2, [300, 1, 129, 200]
    B = len(lens)
    qkv = make_qkv(L, B, H, 77, dtype=torch.float32).cuda()
    lengths = torch.tensor(lens, dtype=torch.int32, device="cuda")
    full = ops.attention_f32(qkv, lengths, L, B, H, True).view(L, B, H * 64)
    out = torch.full((L * B, H * 64), -3.5, device="cuda")
    ops.attention_f32(qkv, lengths, L, B, H, True, out=out,
                      q_limit=torch.tensor([limit], dtype=torch.int32, device="cuda"))
    torch.cuda.synchronize()
    o = out.view(L, B, H * 64)
    q0_lim = _ceil(limit, 128) * 128  # first row of the first tile left untouched
    assert torch.equal(o[:q0_lim], full[:q0_lim])
    assert bool((o[q0_lim:] == -3.5).all())
    pad = padded_tiles(L, B, lens, o.device)
    assert bool((o[:q0_lim][pad[:q0_lim]] == 0).all())
    check_against_ref(full.view(L * B, -1), qkv, L, B, H, lens, True, 77)


@pytest.mark.gpu
def test_attention_f32_head_batch_limit():
    """B*H is a grid dimension: 65535 runs, 65536 is refused (ValueError), not launched."""
    from fbkst_b200 import ops
    L, H = 1, 15
    B = 65535 // H
    qkv = make_qkv(L, B, H, 3, dtype=torch.float32).cuda()
    out = ops.attention_f32(qkv, torch.ones(B, dtype=torch.int32, device="cuda"), L, B, H, True)
    torch.cuda.synchronize()
    v = qkv.view(B, 3, H * 64)[:, 2]
    assert max_norm_err(out.cpu(), v.cpu()) <= TOL_F32  # one key: the output is its value
    H, B = 16, 4096
    qkv = torch.zeros(B, 3 * H * 64, device="cuda")
    with pytest.raises(ValueError):
        ops.attention_f32(qkv, torch.ones(B, dtype=torch.int32, device="cuda"), L, B, H, True)


# --------------------------------------------------------------------------------- cross-attention, S_max
def _xattn_ref(q, kv, mask, row_map, S, U, bsz, tgt, H):
    D = 64 * H
    qd = q.double().cpu().view(tgt, bsz, H, 64)
    kvd = kv.double().cpu()
    rm = row_map.long().cpu()
    k = kvd[:, :, :D].view(S, U, H, 64)[:, rm]
    v = kvd[:, :, D:].view(S, U, H, 64)[:, rm]
    s = torch.einsum("tbhd,sbhd->hbts", qd, k)
    s = s.masked_fill(mask.cpu()[rm].view(1, bsz, 1, S), float("-inf"))
    p = torch.softmax(s, dim=-1)
    return torch.einsum("hbts,sbhd->tbhd", p, v).reshape(tgt * bsz, D), p.mean(0)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_xattn_at_shared_memory_limit(precision):
    """The longest source the cross-attention kernel keeps in shared memory, and the first one it refuses."""
    from fbkst_b200 import ops
    fn, dtype, (tol_o, tol_w) = ((ops.xattn, torch.bfloat16, TOL_XATTN) if precision == "bf16" else
                                 (ops.xattn_f32, torch.float32, TOL_XATTN_F32))
    S, U, bsz, tgt, H = XATTN_S_MAX, 2, 3, 2, 2
    g = torch.Generator().manual_seed(S)
    q = (torch.randn(tgt * bsz, 64 * H, generator=g) * Q_SCALE).to(dtype).cuda()
    kv = torch.randn(S, U, 2 * 64 * H, generator=g).to(dtype).cuda()
    row_map = torch.tensor([1, 0, 1], dtype=torch.int32, device="cuda")
    mask = (torch.arange(S)[None, :] >= torch.tensor([S, S - 1001])[:, None]).cuda()
    out, w = fn(q, kv, mask, row_map, S, U, bsz, tgt, H, weights=1)
    torch.cuda.synchronize()
    ref_o, ref_w = _xattn_ref(q, kv, mask, row_map, S, U, bsz, tgt, H)
    assert max_norm_err(out.cpu(), ref_o) <= tol_o
    assert (w.double().cpu() - ref_w).abs().max().item() <= tol_w
    S += 1
    kv = torch.zeros(S, U, 2 * 64 * H, dtype=dtype, device="cuda")
    mask = torch.zeros(U, S, dtype=torch.bool, device="cuda")
    with pytest.raises(ValueError, match="too long"):
        fn(q, kv, mask, row_map, S, U, bsz, tgt, H, weights=1)


# ------------------------------------------------------------------------------ the bound can see mistakes
MUTANTS = {
    "one key dropped": (lambda n: n - 1, log_penalty),
    "one padding key attended": (lambda n: n + 1, log_penalty),
    "penalty ln(d + 1)": (lambda n: n, torch.log1p),
    "penalty in log2": (lambda n: n, lambda d: torch.log2(d).clamp_min(0)),
    "last 64-key tile dropped": (lambda n: 64 * ((n - 1) // 64), log_penalty),
    "last 128-key tile dropped": (lambda n: 128 * ((n - 1) // 128), log_penalty),
}


def test_reference_sees_mistakes():
    """On the inputs of the host-generated GPU cases with the penalty (short enough to run here), each of these
    kernel mistakes moves some utterance at least 3x TOL_BF16 away from the fp64 reference."""
    worst = dict.fromkeys(MUTANTS, 0.0)
    for case in CASES:
        name, L, B, H, lens, pen, where = resolve(case, sms=148)
        if where != "cpu" or not pen or L > 3000:
            continue
        seed = L * 31 + B * 7 + H
        qkv = make_qkv(L, B, H, seed)
        for b, n in enumerate(lens):
            rows = sample_rows(n, seed + b)
            q, k, v = utterance_operands(qkv, L, B, H, b, rows, min(n + 1, L))
            ref = attn_ref(q, k, v, rows, n, True)
            for m, (keys, penalty) in MUTANTS.items():
                nk = keys(n)
                if 0 < nk <= L:  # a mistake that leaves keys to attend to
                    worst[m] = max(worst[m], max_norm_err(attn_ref(q, k, v, rows, nk, True, penalty), ref))
    print("\n" + "\n".join("%-26s %.3g" % kv for kv in worst.items()))
    for m, e in worst.items():
        assert e >= 3 * TOL_BF16, (m, e)
