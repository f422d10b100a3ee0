"""Per-kernel timing of the HBM-bound kernels at the cfg2 shapes (CUDA events on the launching
stream; a 256 MB L2 flush is queued before every launch, which also keeps the GPU behind the CPU so
that no launch gap leaks into the event interval).  usage: bench_small.py [reps] [name]"""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "fbk-fairseq-st_b200"))
import bench  # noqa: E402
from fbkst_b200 import ops  # noqa: E402

d = torch.device("cuda:0")
flush = torch.empty(256 << 20, dtype=torch.uint8, device=d)
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 10
only = sys.argv[2] if len(sys.argv) > 2 else None
HBM = bench.peaks()["hbm"]
try:  # a time is only worth something with the card and the power limit it was measured at
    _smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    _smi = "nvidia-smi unavailable"
print("device: %s | %s" % (torch.cuda.get_device_name(d), _smi), flush=True)


def timeit(name, fn, nbytes):
    if only and only not in name:
        return
    ts = []
    for i in range(reps + 2):
        flush.fill_(i)
        flush.view(torch.int32).sum()  # read pass: leaves CLEAN lines in L2 (no write-back under the kernel)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    ts = sorted(ts[2:])
    med = ts[len(ts) // 2]
    print("%-26s %8.1f us  %7.0f GB/s  %5.1f%% of %.0f  (min %.1f us)" %
          (name, med * 1e3, nbytes / med / 1e6, 100 * nbytes / med / 1e6 / HBM, HBM, ts[0] * 1e3), flush=True)


def warm_us(fn, n=20, replays=5):
    """Device time per call of ``fn`` with its operands L2-resident: n back-to-back calls captured in one CUDA
    graph, so the host launch path is not what is timed."""
    fn()
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for _ in range(n):
            fn()
    gr.replay()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(replays):
        gr.replay()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / (n * replays) * 1e3


B, T, F, L, D, V = 64, 1500, 40, 375, 512, 8005
lens = torch.full((B,), L, dtype=torch.int32, device=d)
x = torch.randn(B, T, F, device=d)
tl = torch.full((B,), T, dtype=torch.int32, device=d)
timeit("cmvn", lambda: ops.cmvn(x, tl), x.numel() * 4 * 3)

C = 64
w1, b1 = torch.randn(C, 9, device=d), torch.randn(C, device=d)
sc, sh = torch.rand(C, device=d) + 0.5, torch.randn(C, device=d)
y1 = ops.conv1_relu_bn(x, w1, b1, sc, sh)
timeit("conv1", lambda: ops.conv1_relu_bn(x, w1, b1, sc, sh), x.numel() * 4 + y1.numel() * 2)
w2 = ops.prep_conv2_weight(torch.randn(C, C, 3, 3, device=d) * 0.05)
y2 = ops.conv2_relu_bn(y1, w2, b1, sc, sh)
timeit("conv2", lambda: ops.conv2_relu_bn(y1, w2, b1, sc, sh), y1.numel() * 2 + y2.numel() * 2)

p1 = ops.conv1_relu_bn_planes(x, w1, b1, sc, sh)
timeit("conv1 planes", lambda: ops.conv1_relu_bn_planes(x, w1, b1, sc, sh), x.numel() * 4 + p1.numel() * 2)
timeit("conv2 planes", lambda: ops.conv2_relu_bn_planes(p1, y1.shape[1], y1.shape[2], w2, b1, sc, sh),
       p1.numel() * 2 + y2.numel() * 2)

xr = torch.randn(L * B, D, device=d)
g, b_ = torch.randn(D, device=d), torch.randn(D, device=d)
timeit("layernorm f32->bf16", lambda: ops.layernorm(xr, g, b_), xr.numel() * 6)

plan = bench.label_plan(L, B, V, seed=7).to(d)
ldv = (V + 7) // 8 * 8
logits = torch.randn(L * B, ldv, device=d).bfloat16()
logits[:, :V].view(L, B, V).scatter_add_(2, plan.unsqueeze(-1), torch.full((L, B, 1), 30.0, dtype=torch.bfloat16, device=d))
lg = logits[:, :V]
for want in (False, True):
    timeit("ctc_argmax prob=%d" % want, lambda: ops.ctc_argmax(lg, lens, L, B, V, want), L * B * V * 2 + L * B * 8)
for strat in ("avg", "weighted", "softmax"):
    labels, prob = ops.ctc_argmax(lg, lens, L, B, V, True)
    timeit("ctc_segment " + strat, lambda: ops.ctc_segment(labels, prob, lens, strat, L, B), L * B * 20)
    seg_id, seg_start, weight, new_len, max_new = ops.ctc_segment(labels, prob, lens, strat, L, B)
    out = torch.zeros(L * B, D, device=d)
    nl = int(new_len.sum())
    timeit("ctc_compress " + strat, lambda: ops.ctc_compress(xr, seg_id, seg_start, weight, lens, new_len, max_new, L, B, out=out),
           (L * B + nl) * D * 4)
print("compression ratio %.3f" % (nl / (L * B)))

# next row N1: criterion kernels at the cfg2 shape (latency-bound: B CTAs, O(L) dependent steps)
U = 60
tgt = torch.randint(0, V - 1, (B, U), device=d)
tlen = torch.randint(20, U + 1, (B,), device=d).to(torch.int32)
labels, lse, _ = ops.ctc_argmax_lse(lg, lens, L, B, V)
timeit("crit ctc_argmax_lse", lambda: ops.ctc_argmax_lse(lg, lens, L, B, V), L * B * V * 2 + L * B * 8)
timeit("crit ctc_loss_fwd", lambda: ops.ctc_loss_fwd(lg, lse, lens, tgt, tlen, V - 1, L, B, V), L * B * (U + 1) * 2)
timeit("crit ctc_uer", lambda: ops.ctc_uer(labels, lens, tgt, tlen, V - 1, L, B), L * B * 4)

# next row N4: one decoder step of encoder-decoder attention at the cfg2 generate shape (64 utterances
# x beam 5, compressed S = 95, D 512, H 8).  Algorithmic bytes = the UNIQUE K/V (S*U*2D bf16) + q + out;
# the reference's per-hypothesis cache would move bsz*2*S*D fp32 for the same step (printed for scale).
if not only or "xattn" in only:
    for S_, U_, beam_, H_ in ((95, 64, 5, 8), (375, 64, 5, 8), (1500, 8, 5, 16)):
        D_ = 64 * H_
        bsz_ = U_ * beam_
        q_ = torch.randn(bsz_, D_, device=d).bfloat16()
        kv_ = torch.randn(S_, U_, 2 * D_, device=d).bfloat16()
        rm_ = torch.arange(U_, device=d).repeat_interleave(beam_).int()
        mk_ = (torch.arange(S_, device=d)[None, :] >= torch.randint(S_ // 2, S_ + 1, (U_, 1), device=d))
        nb = kv_.numel() * 2 + q_.numel() * 4
        timeit("xattn S=%d U=%d beam=%d H=%d" % (S_, U_, beam_, H_),
               lambda: ops.xattn(q_, kv_, mk_, rm_, S_, U_, bsz_, 1, H_, weights=0), nb)
        timeit("xattn + head-avg weights", lambda: ops.xattn(q_, kv_, mk_, rm_, S_, U_, bsz_, 1, H_, weights=1),
               nb + bsz_ * S_ * 4 * (2 * H_ + 1))
        if not only or "xattn" in only:
            # decode re-reads the same K/V every step: the steady state is L2-resident, not cold
            w_us = warm_us(lambda: ops.xattn(q_, kv_, mk_, rm_, S_, U_, bsz_, 1, H_, weights=0))
            print("    warm (graph of 20 back-to-back steps, K/V L2-resident): %.1f us/step, %.0f GB/s of K/V" %
                  (w_us, nb / w_us / 1e3))
        print("    (reference cache traffic for the step: %.1f MB fp32; unique K/V here: %.1f MB bf16)" %
              (bsz_ * 2 * S_ * D_ * 4 / 1e6, kv_.numel() * 2 / 1e6))

    # the fp32 decode path (CrossAttention.precision = "fp32") against bf16 at the cfg2 generate shape: the core
    # alone, one module call per layer-step (q projection + core + out_proj, no weights, K/V cached) and the
    # once-per-utterance K/V projection.  Bytes: unique K/V + q + out, plus the weights each projection reads.
    from fbkst_b200.cross_attention import CrossAttention
    S_, U_, beam_, H_ = 95, 64, 5, 8
    D_ = 64 * H_
    bsz_ = U_ * beam_
    rm_ = torch.arange(U_, device=d).repeat_interleave(beam_).int()
    mk_ = (torch.arange(S_, device=d)[None, :] >= torch.randint(S_ // 2, S_ + 1, (U_, 1), device=d))
    q32 = torch.randn(bsz_, D_, device=d) * 0.125
    kv32 = torch.randn(S_, U_, 2 * D_, device=d)
    nb32 = kv32.numel() * 4 + q32.numel() * 8
    timeit("xattn f32 S=%d U=%d beam=%d H=%d" % (S_, U_, beam_, H_),
           lambda: ops.xattn_f32(q32, kv32, mk_, rm_, S_, U_, bsz_, 1, H_, weights=0), nb32)
    w_us = warm_us(lambda: ops.xattn_f32(q32, kv32, mk_, rm_, S_, U_, bsz_, 1, H_, weights=0))
    print("    warm (graph of 20 back-to-back steps, K/V L2-resident): %.1f us/step, %.0f GB/s of K/V" %
          (w_us, nb32 / w_us / 1e3))
    enc_ = torch.randn(S_, U_, D_, device=d)
    mpad_ = mk_.view(U_, S_)
    xq_ = torch.randn(1, bsz_, D_, device=d)
    for prec, esz in (("bf16", 2), ("fp32", 4)):
        m_ = CrossAttention(D_, H_).eval().to(d)
        m_.precision = prec
        inc_ = {}
        with torch.no_grad():
            m_(xq_[:, :U_], enc_, enc_, key_padding_mask=mpad_, incremental_state=inc_, static_kv=True)
        m_.reorder_incremental_state(inc_, rm_.long())  # x beam: the row map gathers, the K/V stays per utterance
        step = lambda: m_(xq_, None, None, incremental_state=inc_, static_kv=True, need_weights=False)
        nbm = S_ * U_ * 2 * D_ * esz + 2 * D_ * D_ * esz + bsz_ * D_ * 8
        timeit("xattn module %s step" % prec, step, nbm)
        w_us = warm_us(step)
        print("    warm (graph of 20 back-to-back steps, K/V L2-resident): %.1f us/step" % w_us)
        timeit("xattn module %s K/V proj" % prec, lambda: m_._project_kv(enc_, mpad_, U_),
               enc_.numel() * 4 + 2 * D_ * D_ * esz + S_ * U_ * 2 * D_ * esz)
