"""Training self-attention (csrc/attention_train.cu) at its length, tile and dispatch limits, against fp64.

``ops.attention_train_fwd`` runs the FWD kernel (pass A: exact row LSE; pass B: P = 2^(s - LSE), dropout,
O += P V); ``ops.attention_train_bwd`` runs ``fbkst_attn_delta`` and then the DQ kernel (own rows = queries) and
the DKV kernel (own rows = keys, so padded queries are handled from the other side).  Each CTA owns 128 rows and
walks the other side in 64-row tiles.  The cases sit where such kernels go wrong: a lone key tile, odd and even
key-tile counts (the FWD main pass starts its TMA stages at ``n_oth & 1``), utterances of length 1, query and key
tiles made only of padding inside a longer batch, 16 heads (D = 1024), cfg4's B * H = 512, the last L at two CTAs
per SM, the largest L the shared-memory LUT allows, and the B * H grid limit.  Dropout is checked against a host
restatement of the mask, bit for bit, from the side of each of the three kernels.

The reference is fp64 on the kernel's own bf16 operands, computed over every valid row and compared on every
valid row: O and the log2-domain LSE of each query, dQ of each query and dK / dV of each key.  The backward's
operands include the forward output it is given: delta = rowsum(dO o O) is formed from that stored bf16 O, by the
kernels and by the reference alike.  With the exact O instead, the gradients would also carry O's bf16 rounding,
2^-9 of sum |dO| |O|, which is not small against dP o keep - delta where that difference cancels (one frame,
dropout, dO . v = 0.32 with sum |dO| |O| = 47: 2.4e-2 on a B200, reproduced exactly by emulating the roundings
on the host).  O itself is checked against the exact fp64 forward.  Errors are per
(utterance, head).  O is max-normalised; the LSE error is absolute; a gradient's error is divided by the largest
value of the same sum taken over the magnitudes of its terms (dQ: |dS| bound @ |K| with |dS| <= P (|dP o keep| +
|delta|) scale; dK: the same with |Q|; dV: (P o keep)^T |dO|).  That is the scale a bf16 rounding of the terms
errs by; it stays finite where dP - delta cancels, e.g. dQ = dK = 0 exactly for an utterance of one frame.

Scores have std 3 (q scaled by Q_SCALE before the kernel's 1/8), so the mask, the penalty and dropout change the
result.  ``test_reference_sees_mistakes`` (no GPU) shows that these bounds see the mistakes the kernels could make
at these edges.

The bounds in TOL are the starting ones: 8e-3 for O (bf16 output rounding plus the bf16 P, as in the inference
edge tests), 1e-3 on the log2 LSE and 2e-2 for the gradients.  The worst errors on a B200 have not been measured
yet; once they are, each bound belongs at about 3x the measured worst.  On the short cases every mutant is at least
20x its tolerance away, so tightening the bounds that far leaves the mutant test its margin."""
import math

import numpy as np
import pytest
import torch

Q_SCALE = 3.0          # q before the kernel's 0.125: scores of std 3
SCALE = 0.125          # head_dim ** -0.5
LOG2E = 1.0 / math.log(2.0)
TOL = {"o": 8e-3, "lse": 1e-3, "dq": 2e-2, "dk": 2e-2, "dv": 2e-2}
SEED, SITE = 987654321, 3


def _ceil(a, b):
    return -(-a // b)


# ---------------------------------------------------------------------------------- host-side restatement
# attn_train_smem: Q/K, dO/V (2 x 16 KB), two stages of two 8 KB other-side tiles, two written 16 KB tiles,
# 64 B of barriers, the (lse, delta) and (m, l) exchange buffers, 1 KB of alignment slack, and the penalty LUT
# of 2 * ceil(L / 128) * 128 floats.
SMEM_MAX = 227 * 1024       # per CTA
SMEM_SM = 228 * 1024        # per SM (1 KB of it reserved per resident CTA)
TR_SMEM_FIXED = 2 * 16384 + 4 * 8192 + 2 * 16384 + 64 + 4 * 128 * 2 + 4 * 512 + 1024


def train_smem(L):
    return TR_SMEM_FIXED + 8 * _ceil(L, 128) * 128


def ctas_per_sm(L):
    return SMEM_SM // (train_smem(L) + 1024)


L_MAX = 16128


def test_shared_memory_limits():
    assert TR_SMEM_FIXED == 102464
    assert max(L for L in range(1, 20000) if train_smem(L) <= SMEM_MAX) == L_MAX
    assert train_smem(L_MAX + 1) > SMEM_MAX
    assert _ceil(L_MAX, 64) == 252 and _ceil(L_MAX, 128) == 126
    # __launch_bounds__(256, 2): two CTAs per SM while their shared memory fits, one beyond
    assert max(L for L in range(1, L_MAX + 1) if ctas_per_sm(L) >= 2) == 1536
    assert ctas_per_sm(1) == 2 and ctas_per_sm(1537) == 1 and ctas_per_sm(L_MAX) == 1


# Dropout: keep (q, k) of head-batch bh iff lowbias32(q A ^ k B ^ bh C ^ key) >= threshold, key = mix_key(seed, site)
M64 = (1 << 64) - 1


def mix_key(seed, site):
    x = (seed ^ (0x9E3779B97F4A7C15 * ((site + 1) & M64))) & M64
    x ^= x >> 33
    x = (x * 0xFF51AFD7ED558CCD) & M64
    x ^= x >> 33
    return (x ^ (x >> 32)) & 0xFFFFFFFF


def drop_threshold(p):
    p = np.float32(p)
    if not p > 0:
        return 0
    t = float(p) * 4294967296.0
    return max(1, 0xFFFFFFFF if t >= 4294967295.0 else int(t))


def drop_scale(p):
    return float(np.float32(1.0) / (np.float32(1.0) - np.float32(p))) if p > 0 else 1.0


def tr_keep(key, threshold, bh, q, k):
    """Keep flags (bool) of broadcastable uint32-able index arrays bh, q, k."""
    u = np.uint32
    bh, q, k = (np.asarray(a, dtype=np.uint32) for a in (bh, q, k))
    x = (q * u(0x9E3779B1)) ^ (k * u(0x85EBCA77)) ^ (bh * u(0xC2B2AE3D)) ^ u(key)
    x ^= x >> u(16)
    x *= u(0x7FEB352D)
    x ^= x >> u(15)
    x *= u(0x846CA68B)
    x ^= x >> u(16)
    return x >= u(threshold)


def keep_mask(p, seed, site, BH, L):
    """[BH, L, L] keep-scale (0 or 1 / (1 - p)) as fp64, or None without dropout."""
    if p == 0:
        return None
    keep = tr_keep(mix_key(seed, site), drop_threshold(p), np.arange(BH)[:, None, None], np.arange(L)[None, :, None],
                   np.arange(L)[None, None, :])
    return torch.from_numpy(keep).double() * drop_scale(p)


def test_drop_threshold():
    assert drop_threshold(0.0) == 0
    assert drop_threshold(0.5) == 1 << 31
    assert drop_threshold(0.1) == 429496736  # float32(0.1) * 2^32, exactly
    assert drop_threshold(1e-12) == 1        # a tiny p still drops something
    assert drop_threshold(np.nextafter(np.float32(1), np.float32(0))) == 4294967040
    assert drop_scale(0.25) == float(np.float32(1) / np.float32(0.75))


def _chi2_ok(kept, n, r):
    """Group counts ``kept`` out of ``n`` at keep rate r look binomial: neither too spread nor too even."""
    from scipy.stats import chi2
    stat = float((((kept - n * r) ** 2) / (n * r * (1 - r))).sum())
    dof = kept.size
    return chi2.sf(stat, dof) > 1e-6 and chi2.cdf(stat, dof) > 1e-6, (stat, dof)


@pytest.mark.parametrize("p", [0.1, 0.25, 0.5])
def test_dropout_hash_statistics(p):
    BH, L = 6, 384
    key, thr = mix_key(SEED, SITE), drop_threshold(p)
    bh, q, k = np.arange(BH)[:, None, None], np.arange(L)[None, :, None], np.arange(L)[None, None, :]
    keep = tr_keep(key, thr, bh, q, k)
    r = 1.0 - thr / 2.0 ** 32
    N = keep.size
    assert abs(keep.mean() - r) <= 5 * math.sqrt(r * (1 - r) / N), keep.mean()
    ok, info = _chi2_ok(keep.sum(2).ravel(), L, r)
    assert ok, ("rows", info)
    ok, info = _chi2_ok(keep.sum(1).ravel(), L, r)
    assert ok, ("columns", info)
    # diagonals k - q = d of at least 32 elements
    kept, n = [], []
    for d in range(-(L - 32), L - 31):
        dg = np.diagonal(keep, offset=d, axis1=1, axis2=2)
        kept += dg.sum(1).tolist()
        n += [dg.shape[1]] * BH
    ok, info = _chi2_ok(np.array(kept), np.array(n), r)
    assert ok, ("diagonals", info)
    # the position inside a 64 x 64 tile, and the head-batch
    ok, info = _chi2_ok(keep.reshape(BH, L // 64, 64, L // 64, 64).sum((0, 1, 3)).ravel(), BH * (L // 64) ** 2, r)
    assert ok, ("tile position", info)
    ok, info = _chi2_ok(keep.sum((1, 2)), L * L, r)
    assert ok, ("head-batch", info)
    # another site, another seed, another head, the transpose: independent masks agree on r^2 + (1 - r)^2
    agree = r * r + (1 - r) ** 2
    others = {"site": tr_keep(mix_key(SEED, SITE + 1), thr, bh, q, k),
              "seed": tr_keep(mix_key(SEED + 1, SITE), thr, bh, q, k),
              "seed + 2^32": tr_keep(mix_key(SEED + (1 << 32), SITE), thr, bh, q, k),
              "head": tr_keep(key, thr, bh + 1, q, k),
              "transpose": keep.transpose(0, 2, 1)}
    for name, other in others.items():
        a = (other == keep).mean()
        assert abs(a - agree) <= 5 * math.sqrt(agree * (1 - agree) / N), (name, a, agree)


# ------------------------------------------------------------------------------------------ fp64 reference
def log_penalty(d):
    return torch.log(d).clamp_min(0)  # ln(max(1, |i - j|)), 0 on the diagonal


MUTANTS = ["dq drops the last 64-key tile", "dk/dv drop the last 64-query tile", "one padding key attended",
           "keep transposed in dk/dv", "delta from the undropped output", "penalty ln(d + 1)"]


def attn_train_ref(q, k, v, do, n, pen, keep=None, o_fwd=None, mutant=None, chunk=512):
    """fp64 forward and backward of one utterance (all heads) on the kernel's operands.

    q, k, v, do: [>= n, H, 64], q unscaled as the kernel reads it; rows from n on are padding.  keep: [H, >= n, >= n]
    keep-scale of the dropout mask, or None.  o_fwd: [>= n, H, 64], the stored forward output that the backward
    takes as an input and forms delta = rowsum(dO o O) from; None stands for the fp64 O rounded to bf16, as the
    forward stores it.  Query rows are processed in chunks, so L = 16128 fits in memory.
    Returns a dict of [H, n, 64] fp64 tensors o, dq, dk, dv and their term magnitudes mo, mdq, mdk, mdv, and lse
    [H, n] in the kernel's log2 domain.  ``mutant`` (one of MUTANTS) computes a deliberately wrong variant."""
    nk = n + 1 if mutant == "one padding key attended" else n
    penalty = torch.log1p if mutant == "penalty ln(d + 1)" else log_penalty
    cut = 64 * ((n - 1) // 64)  # first row of the last 64-row tile
    Q, K, V, dO = (x.double().permute(1, 0, 2) for x in (q[:n], k[:nk], v[:nk], do[:n]))  # [H, rows, 64]
    Of = None if o_fwd is None else o_fwd[:n].double().permute(1, 0, 2)
    H, dev = Q.shape[0], Q.device
    keys = torch.arange(nk, device=dev)
    r = {name: torch.zeros(H, n, 64, dtype=torch.float64, device=dev) for name in ("o", "dq", "mdq")}
    r["lse"] = torch.zeros(H, n, dtype=torch.float64, device=dev)
    for name in ("dk", "dv", "mdk", "mdv"):
        r[name] = torch.zeros(H, nk, 64, dtype=torch.float64, device=dev)
    for c0 in range(0, n, chunk):
        c1 = min(c0 + chunk, n)
        Qc, dOc = Q[:, c0:c1], dO[:, c0:c1]
        s = Qc @ K.transpose(1, 2) * SCALE
        if pen:
            s = s - penalty((torch.arange(c0, c1, device=dev)[:, None] - keys[None, :]).abs().double())
        lse = torch.logsumexp(s, -1, keepdim=True)
        P = torch.exp(s - lse)
        kp = keep[:, c0:c1, :nk] if keep is not None else torch.ones_like(P)
        O = (P * kp) @ V
        dP = dOc @ V.transpose(1, 2)
        if mutant == "delta from the undropped output":
            stored = P @ V
        else:
            stored = O.bfloat16().double() if Of is None else Of[:, c0:c1]
        delta = (dOc * stored).sum(-1, keepdim=True)
        dS = P * (dP * kp - delta) * SCALE
        mS = P * ((dP * kp).abs() + delta.abs()) * SCALE
        r["o"][:, c0:c1], r["lse"][:, c0:c1] = O, lse[..., 0] * LOG2E
        if mutant == "dq drops the last 64-key tile":
            r["dq"][:, c0:c1] = dS[..., :cut] @ K[:, :cut]
        else:
            r["dq"][:, c0:c1] = dS @ K
        r["mdq"][:, c0:c1] = mS @ K.abs()
        if mutant == "keep transposed in dk/dv":
            kp = keep[:, :nk, c0:c1].transpose(1, 2)
            dS = P * (dP * kp - delta) * SCALE
        if mutant == "dk/dv drop the last 64-query tile":
            w = (torch.arange(c0, c1, device=dev) < cut).double()[None, :, None]
            dS, kp = dS * w, kp * w
        r["dk"] += dS.transpose(1, 2) @ Qc
        r["dv"] += (P * kp).transpose(1, 2) @ dOc
        r["mdk"] += mS.transpose(1, 2) @ Qc.abs()
        r["mdv"] += (P * kp).transpose(1, 2) @ dOc.abs()
    r["mo"] = r["o"]
    for name in ("dk", "dv", "mdk", "mdv"):
        r[name] = r[name][:, :n]
    return r


def head_errors(got, ref):
    """{quantity: [H] errors} of got (dict of [H, n, ...] tensors) against the reference dict."""
    e = {}
    for name in ("o", "dq", "dk", "dv"):
        a, b = got[name].double().to(ref[name].device), ref[name]
        diff = (a - b).abs().flatten(1).max(1).values
        e[name] = diff / ref["m" + name].abs().flatten(1).max(1).values.clamp_min(1e-300)
        e[name] = torch.where(torch.isfinite(a).flatten(1).all(1), e[name], torch.full_like(e[name], math.inf))
    e["lse"] = (got["lse"].double().to(ref["lse"].device) - ref["lse"]).abs().max(1).values
    return {k: v.cpu() for k, v in e.items()}


# ------------------------------------------------------------------------------------------ inputs, cases
def make_inputs(L, B, H, seed, device="cpu"):
    """qkv [L*B, 3*H*64] bf16 (row t*B + b, q scaled by Q_SCALE) and dO [L*B, H*64] bf16, random on every row."""
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.randn(L * B, 3 * H * 64, generator=g, device=device)
    x[:, : 64 * H] *= Q_SCALE
    do = torch.randn(L * B, H * 64, generator=g, device=device)
    return x.bfloat16(), do.bfloat16()


def utterance(qkv, do, L, B, H, b, device):
    """(q, k, v, do) of utterance b, each [L, H, 64], on ``device``."""
    x = qkv.view(L, B, 3, H, 64)[:, b].to(device)
    return x[:, 0], x[:, 1], x[:, 2], do.view(L, B, H, 64)[:, b].to(device)


def kernel_rows(out, lse, dqkv, L, B, H, b, n):
    g = dqkv.view(L, B, 3, H, 64)[:n, b]
    return {"o": out.view(L, B, H, 64)[:n, b].permute(1, 0, 2), "lse": lse.view(B, H, L)[b, :, :n],
            "dq": g[:, 0].permute(1, 0, 2), "dk": g[:, 1].permute(1, 0, 2), "dv": g[:, 2].permute(1, 0, 2)}


def _ragged(L):
    """1, L, L - 1 and the multiples of 64 and 128 +-1 below L: a lone key tile, partial key tiles, and query
    tiles wholly beyond the length."""
    lens = {1, L, max(L - 1, 1)}
    for m in (64, 128, 256):
        lens.update(x for x in (m - 1, m, m + 1) if x <= L)
    return sorted(lens, reverse=True)


def _cases():
    """(id, L, B, H, lengths, penalty, dropout p)."""
    cases = []
    for i, L in enumerate([1, 2, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 257]):
        for H in (1, 3, 16):
            pen = (i + H) % 2 == 0
            lens = _ragged(L)
            cases.append(("L%d_H%d_%s" % (L, H, "pen" if pen else "nopen"), L, len(lens), H, lens, pen, 0.0))
    ctc = [283, 271, 240, 201, 180, 150, 129, 128, 100, 77, 64, 50, 31, 17, 5, 1]
    cases += [
        ("cfg4_375", 375, 64, 8, [375] * 64, True, 0.0),          # 64 x 1500 frames after the 4x subsampling
        ("ctc_283", 283, 16, 8, ctc, True, 0.0),                  # after CTC compression: ragged, L % 8 != 0
        ("ctc_283_nopen", 283, 16, 8, ctc, False, 0.0),
        ("two_cta_1536", 1536, 3, 2, [1536, 1473, 700], True, 0.0),
        ("one_cta_1537", 1537, 3, 2, [1537, 1536, 65], False, 0.0),
        ("longest_16128", L_MAX, 3, 1, [L_MAX, 16065, 1], True, 0.0),
        ("drop0.1_pen", 300, 5, 3, [300, 257, 129, 64, 1], True, 0.1),
        ("drop0.1_nopen", 300, 5, 3, [300, 257, 129, 64, 1], False, 0.1),
        ("drop0.5_pen", 193, 4, 5, [193, 192, 65, 2], True, 0.5),
        ("drop0.5_nopen", 193, 4, 5, [193, 192, 65, 2], False, 0.5),
    ]
    return cases


CASES = _cases()


def _ref_device(L, B, H):
    return "cuda" if L * L * B * H > 2e7 else "cpu"


def padded_tiles(L, B, lens, device):
    """[L, B] bool: rows of 128-row tiles that lie wholly beyond the utterance's length."""
    start = torch.tensor([_ceil(n, 128) * 128 for n in lens], device=device)
    return torch.arange(L, device=device)[:, None] >= start[None, :]


def padded_rows(L, B, lens, device):
    return torch.arange(L, device=device)[:, None] >= torch.tensor(lens, device=device)[None, :]


def run_kernels(qkv, do, lengths, L, B, H, pen, p):
    from fbkst_b200 import ops
    out, lse = ops.attention_train_fwd(qkv, lengths, L, B, H, pen, p=p, seed=SEED, site=SITE)
    dqkv = ops.attention_train_bwd(qkv, out, do, lse, lengths, L, B, H, pen, p=p, seed=SEED, site=SITE)
    return out, lse, dqkv


# ------------------------------------------------------------------------------------------------- GPU cases
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_attention_train_vs_fp64(case):
    name, L, B, H, lens, pen, p = case
    assert len(lens) == B and max(lens) <= L
    seed = L * 31 + B * 7 + H
    qkv, do = (x.cuda() for x in make_inputs(L, B, H, seed))
    lengths = torch.tensor(lens, dtype=torch.int32, device="cuda")
    out, lse, dqkv = run_kernels(qkv, do, lengths, L, B, H, pen, p)
    again = run_kernels(qkv, do, lengths, L, B, H, pen, p)
    torch.cuda.synchronize()
    for a, b, what in zip((out, lse, dqkv), again, ("O", "LSE", "dqkv")):
        assert torch.equal(a, b), "two identical calls differ: " + what
    tiles = padded_tiles(L, B, lens, "cuda")
    assert bool((out.view(L, B, -1)[tiles] == 0).all()), "O of padded query tiles is not zero"
    assert bool((lse.view(B, H, L).permute(2, 0, 1)[tiles] == 0).all()), "LSE of padded query tiles is not zero"
    assert bool((dqkv.view(L, B, -1)[padded_rows(L, B, lens, "cuda")] == 0).all()), "padded rows have gradients"
    dev = _ref_device(L, B, H)
    keep = keep_mask(p, SEED, SITE, B * H, L)
    worst = dict.fromkeys(TOL, 0.0)
    for b, n in enumerate(lens):
        ref = attn_train_ref(*utterance(qkv, do, L, B, H, b, dev), n, pen,
                             None if keep is None else keep[b * H:(b + 1) * H].to(dev),
                             o_fwd=out.view(L, B, H, 64)[:, b].to(dev))
        for q, e in head_errors(kernel_rows(out, lse, dqkv, L, B, H, b, n), ref).items():
            assert bool((e <= TOL[q]).all()), (q, "utterance", b, "length", n, "heads", e.tolist())
            worst[q] = max(worst[q], e.max().item())
    print("\n%s: worst %s" % (name, " ".join("%s %.3g" % kv for kv in worst.items())))


@pytest.mark.gpu
@pytest.mark.parametrize("L,B,H,p,windows", [(300, 2, 3, 0.25, (0, 128, 236)),
                                             (2500, 1, 5, 0.1, (0, 1216, 2436))])
def test_dropout_mask_matches_host(L, B, H, p, windows):
    """The keep mask each kernel applies equals the host restatement, bit for bit.  With q = 0 every probability
    is 1 / L (no penalty), so one-hot probes over a 64-row window read the mask out:
      FWD:  V[w + i] = e_i                        -> O[q, i]  = keep(q, w + i) / L
      DKV:  the same, dO[w + i] = e_i             -> dV[k, i] = keep(w + i, k) / L
      DQ:   K[w + i] = e_i, V[:, 0] = dO[:, 0] = 1 -> dQ[q, i] = (keep(q, w + i) - delta_q) / (8 L),
            delta_q = O[q, 0]."""
    from fbkst_b200 import ops
    D, BH, ds = H * 64, B * H, drop_scale(p)
    lengths = torch.full((B,), L, dtype=torch.int32, device="cuda")
    key, thr = mix_key(SEED, SITE), drop_threshold(p)
    eye = torch.eye(64, device="cuda")
    for w in windows:
        host_k = torch.from_numpy(tr_keep(key, thr, np.arange(BH)[:, None, None], np.arange(L)[None, :, None],
                                          w + np.arange(64)[None, None, :]))          # [BH, q, window keys]
        host_q = torch.from_numpy(tr_keep(key, thr, np.arange(BH)[:, None, None], w + np.arange(64)[None, :, None],
                                          np.arange(L)[None, None, :]))               # [BH, window queries, k]
        qkv = torch.zeros(L, B, 3, H, 64, device="cuda")
        qkv[w:w + 64, :, 2] = eye[:, None, None, :]
        do = torch.zeros(L, B, H, 64, device="cuda")
        do[w:w + 64] = eye[:, None, None, :]
        qkv, do = qkv.view(L * B, 3 * D).bfloat16(), do.view(L * B, D).bfloat16()
        out, lse, dqkv = run_kernels(qkv, do, lengths, L, B, H, False, p)
        o = out.float().view(L, BH, 64).permute(1, 0, 2)                                  # [BH, q, i]
        dv = dqkv.float().view(L, B, 3, H, 64)[:, :, 2].reshape(L, BH, 64).permute(1, 2, 0)  # [BH, i, k]
        assert torch.equal(o.cpu() != 0, host_k), ("FWD", w)
        assert torch.equal(dv.cpu() != 0, host_q), ("DKV", w)
        kept = o[o != 0] * L
        assert torch.allclose(kept, torch.full_like(kept, ds), rtol=1e-2), ("FWD keep scale", w)
        # DQ
        qkv = torch.zeros(L, B, 3, H, 64, device="cuda")
        qkv[w:w + 64, :, 1] = eye[:, None, None, :]
        qkv[:, :, 2, :, 0] = 1
        do = torch.zeros(L, B, H, 64, device="cuda")
        do[..., 0] = 1
        qkv, do = qkv.view(L * B, 3 * D).bfloat16(), do.view(L * B, D).bfloat16()
        out, lse, dqkv = run_kernels(qkv, do, lengths, L, B, H, False, p)
        delta = out.float().view(L, BH, 64)[:, :, 0].t()[:, :, None]                       # [BH, q, 1]
        dq = dqkv.float().view(L, B, 3, H, 64)[:, :, 0].reshape(L, BH, 64).permute(1, 0, 2)
        keep_dq = dq * (L / SCALE) + delta
        assert torch.equal((keep_dq > 0.5 * ds).cpu(), host_k), ("DQ", w)


@pytest.mark.gpu
@pytest.mark.parametrize("pen,p", [(True, 0.0), (False, 0.25)])
def test_padded_rows_do_not_leak(pen, p):
    """qkv and dO rows at or beyond an utterance's length are never read into a valid result: filling them
    with +-3e4 gives bit-identical O, LSE and dqkv on valid rows, and exact zeros on the padded ones."""
    L, H, lens = 300, 2, [300, 129, 65, 1]
    B = len(lens)
    qkv, do = (x.cuda() for x in make_inputs(L, B, H, 11))
    lengths = torch.tensor(lens, dtype=torch.int32, device="cuda")
    pad = padded_rows(L, B, lens, "cuda")
    runs = []
    for fill in ("zero", "big"):
        x, g = qkv.clone().view(L, B, -1), do.clone().view(L, B, -1)
        for t in (x, g):
            if fill == "zero":
                t[pad] = 0
            else:
                t[pad] = (torch.randint(0, 2, t[pad].shape, device="cuda") * 6e4 - 3e4).bfloat16()
        runs.append(run_kernels(x.view(L * B, -1), g.view(L * B, -1), lengths, L, B, H, pen, p))
    torch.cuda.synchronize()
    (o0, l0, d0), (o1, l1, d1) = runs
    valid = ~pad
    assert torch.equal(o0.view(L, B, -1)[valid], o1.view(L, B, -1)[valid])
    lv = valid.t()[:, None, :].expand(B, H, L)
    assert torch.equal(l0.view(B, H, L)[lv], l1.view(B, H, L)[lv])
    assert torch.equal(d0, d1)
    assert bool((d1.view(L, B, -1)[pad] == 0).all())
    tiles = padded_tiles(L, B, lens, "cuda")
    assert bool((o1.view(L, B, -1)[tiles] == 0).all())
    assert bool((l1.view(B, H, L).permute(2, 0, 1)[tiles] == 0).all())


@pytest.mark.gpu
def test_head_batch_limit():
    """B * H is a grid dimension: 65535 runs (one frame: each output row is its value row, dV is dO), 65536 is
    refused with ValueError by the forward and the backward, not launched."""
    from fbkst_b200 import ops
    L, H = 1, 15
    B = 65535 // H
    D = H * 64
    qkv, do = (x.cuda() for x in make_inputs(L, B, H, 3))
    lengths = torch.ones(B, dtype=torch.int32, device="cuda")
    out, lse, dqkv = run_kernels(qkv, do, lengths, L, B, H, True, 0.0)
    torch.cuda.synchronize()
    assert torch.equal(out, qkv[:, 2 * D:])
    assert torch.equal(dqkv[:, 2 * D:], do)
    assert bool(torch.isfinite(dqkv).all()) and dqkv[:, :2 * D].abs().max().item() < 1e-2  # exactly 0 in fp64
    H, B = 16, 4096
    qkv = torch.zeros(B, 3 * H * 64, dtype=torch.bfloat16, device="cuda")
    lengths = torch.ones(B, dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError, match="bad shape"):
        ops.attention_train_fwd(qkv, lengths, L, B, H)
    out = torch.zeros(B, H * 64, dtype=torch.bfloat16, device="cuda")
    lse = torch.zeros(B * H, L, device="cuda")
    with pytest.raises(ValueError, match="bad shape"):
        ops.attention_train_bwd(qkv, out, out, lse, lengths, L, B, H)


@pytest.mark.gpu
def test_refuses_past_the_shared_memory_limit():
    from fbkst_b200 import ops
    L = L_MAX + 1
    qkv = torch.zeros(L, 3 * 64, dtype=torch.bfloat16, device="cuda")
    lengths = torch.tensor([L], dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError, match="shared memory"):
        ops.attention_train_fwd(qkv, lengths, L, 1, 1)
    out = torch.zeros(L, 64, dtype=torch.bfloat16, device="cuda")
    lse = torch.zeros(1, L, device="cuda")
    with pytest.raises(ValueError, match="shared memory"):
        ops.attention_train_bwd(qkv, out, out, lse, lengths, L, 1, 1)


# ------------------------------------------------------------------------------ the bound can see mistakes
def test_reference_sees_mistakes():
    """On the inputs of the short GPU cases with the penalty or dropout, each mutant of the reference moves some
    (utterance, head) at least 3x its tolerance away from the reference in one of O, dQ, dK, dV."""
    worst = dict.fromkeys(MUTANTS, 0.0)
    for name, L, B, H, lens, pen, p in CASES:
        if _ref_device(L, B, H) != "cpu" or not (pen or p):
            continue
        seed = L * 31 + B * 7 + H
        qkv, do = make_inputs(L, B, H, seed)
        keep = keep_mask(p, SEED, SITE, B * H, L)
        for b, n in enumerate(lens):
            ops_ = utterance(qkv, do, L, B, H, b, "cpu")
            kb = None if keep is None else keep[b * H:(b + 1) * H]
            ref = attn_train_ref(*ops_, n, pen, kb)
            for m in MUTANTS:
                if ((m.startswith("dq") or m.startswith("dk")) and n <= 64) or (m.startswith("one") and n == L) or \
                        (m.startswith("penalty") and not pen) or (("keep" in m or "delta" in m) and kb is None):
                    continue  # the mistake changes nothing here, or leaves no key to attend to
                e = head_errors(attn_train_ref(*ops_, n, pen, kb, mutant=m), ref)
                worst[m] = max(worst[m], max(e[q].max().item() / TOL[q] for q in ("o", "dq", "dk", "dv")))
    print("\n" + "\n".join("%-36s %.3g x tol" % kv for kv in worst.items()))
    for m, r in worst.items():
        assert r >= 3, (m, r)
