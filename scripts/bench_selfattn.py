"""Decoder self-attention (DESIGN §7 N5) at the cfg2 generate shape: 64 utterances x beam 5 = 320 hypotheses,
D 512, H 8, at decoder steps t in {32, 96, 192}.  usage: bench_selfattn.py [reps]

  core     fbkst_dec_self_attn_fwd / _f32 alone, keys gathered through a random within-beam ancestry table;
           cold = a 256 MB L2 flush queued before every launch, warm = 20 back-to-back calls in one CUDA graph
  module   one DecoderSelfAttention step: the q|k|v GEMM into the cache slab, the core, out_proj
  torch    the same step on the torch restatement of the reference's incremental path (separate q/k/v F.linear,
           torch.cat append of the fp32 K/V cache, bmm, fp32 softmax, bmm, out_proj) plus the index_select
           beam reorder of the cache that precedes it
  decode   6 layers x 150 steps with one beam reorder per step (ancestry table here, cache gather in the
           restatement), mean ms per step; the other decoder ops are not part of this loop

Times are CUDA-event medians; the bytes printed are computed from shapes."""
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "fbk-fairseq-st_b200"))
from fbkst_b200 import ops  # noqa: E402
from fbkst_b200.self_attention import DecoderSelfAttention  # noqa: E402

d = torch.device("cuda:0")
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
flush = torch.empty(256 << 20, dtype=torch.uint8, device=d)
try:  # a time is only worth something with the card and the power limit it was measured at
    _smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                           "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    _smi = "nvidia-smi unavailable"
print("device: %s | %s" % (torch.cuda.get_device_name(d), _smi), flush=True)

U, BEAM, D, H = 64, 5, 512, 8
BSZ = U * BEAM


def cold_us(fn):
    ts = []
    for i in range(reps + 2):
        flush.fill_(i)
        flush.view(torch.int32).sum()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    ts = sorted(ts[2:])
    return ts[len(ts) // 2] * 1e3


def warm_us(fn, n=20, replays=5):
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


def beam_order(g):
    """A same-size reorder: every hypothesis picks a parent among its own sentence's beam."""
    o = torch.arange(BSZ).view(U, BEAM)
    return o.gather(1, torch.randint(0, BEAM, (U, BEAM), generator=g)).view(-1)


g = torch.Generator().manual_seed(0)
P = {k: torch.randn(D, D, generator=g) * D ** -0.5 for k in ("q", "k", "v", "o")}
P.update({"b" + k: torch.randn(D, generator=g) * 0.1 for k in ("q", "k", "v", "o")})
P = {k: v.to(d) for k, v in P.items()}


def make_module(prec):
    m = DecoderSelfAttention(D, H).eval().to(d)
    with torch.no_grad():
        for nm, k in (("q_proj", "q"), ("k_proj", "k"), ("v_proj", "v"), ("out_proj", "o")):
            getattr(m, nm).weight.copy_(P[k])
            getattr(m, nm).bias.copy_(P["b" + k])
    m.precision = prec
    return m


def torch_step(x, st, order):
    """The reference's incremental self-attention step (multihead_attention.py, self_attention=True) in torch,
    preceded by its reorder_incremental_state gather."""
    if order is not None:
        st["k"], st["v"] = st["k"].index_select(0, order), st["v"].index_select(0, order)
    q = F.linear(x, P["q"], P["bq"]) * 0.125
    k, v = F.linear(x, P["k"], P["bk"]), F.linear(x, P["v"], P["bv"])
    sp = lambda t: t.contiguous().view(1, BSZ * H, 64).transpose(0, 1)
    q, k, v = sp(q), sp(k), sp(v)
    if "k" in st:
        k = torch.cat([st["k"].view(BSZ * H, -1, 64), k], 1)
        v = torch.cat([st["v"].view(BSZ * H, -1, 64), v], 1)
    st["k"], st["v"] = k.view(BSZ, H, -1, 64), v.view(BSZ, H, -1, 64)
    p = torch.softmax(torch.bmm(q, k.transpose(1, 2)).float(), -1)
    a = torch.bmm(p, v).transpose(0, 1).contiguous().view(1, BSZ, D)
    return F.linear(a, P["o"], P["bo"])


with torch.no_grad():
    gd = torch.Generator(device=d).manual_seed(1)
    x = torch.randn(1, BSZ, D, device=d, generator=gd)
    order = beam_order(g).to(d)
    for t in (32, 96, 192):
        print("--- t = %d (keys per query), %d hypotheses" % (t, BSZ), flush=True)
        sent = torch.arange(BSZ, device=d) // BEAM * BEAM
        anc = (sent[None, :] + torch.randint(0, BEAM, (t, BSZ), device=d, generator=gd)).int().contiguous()
        anc[-1] = torch.arange(BSZ, device=d, dtype=torch.int32)
        for prec, dt, fn in (("bf16", torch.bfloat16, ops.dec_self_attn), ("fp32", torch.float32,
                                                                            ops.dec_self_attn_f32)):
            cache = torch.randn(t, BSZ, 3 * D, device=d, generator=gd).to(dt)
            q = cache[t - 1, :, :D]
            core = lambda: fn(q, cache, anc, None, t, BSZ, 1, H)
            kv = BSZ * t * 2 * D * cache.element_size()
            c_us, w_us = cold_us(core), warm_us(core)
            print("core %s   cold %7.1f us  warm %7.1f us  (K/V rows read per step %.1f MB, %.0f GB/s cold)" %
                  (prec, c_us, w_us, kv / 1e6, kv / c_us / 1e3), flush=True)
        for prec in ("bf16", "fp32"):
            m = make_module(prec)
            inc = {}
            for s in range(t):
                m(x, None, None, incremental_state=inc, need_weights=False)
            buf = m._get_input_buffer(inc)

            def step():  # re-runs step t-1 on the same state: same shapes, same cache slab, no growth
                buf["fbkst_steps"] = t - 1
                m(x, None, None, incremental_state=inc, need_weights=False)

            print("module %s step  cold %7.1f us  warm %7.1f us" % (prec, cold_us(step), warm_us(step)), flush=True)
            del inc, buf
        st = {"k": torch.randn(BSZ, H, t - 1, 64, device=d), "v": torch.randn(BSZ, H, t - 1, 64, device=d)}
        k0, v0 = st["k"], st["v"]

        def ref_step():
            st["k"], st["v"] = k0, v0
            torch_step(x, st, order)

        cache_mb = BSZ * D * (t - 1) * 4 / 1e6
        print("torch restatement fp32 step (reorder + cat + attention)  cold %7.1f us  warm %7.1f us  "
              "(one K or V cache %.1f MB; gather + append move ~%.0f MB)" %
              (cold_us(ref_step), warm_us(ref_step), cache_mb, 8 * cache_mb), flush=True)
        del st, k0, v0

    # ---- 6-layer decode loop, 150 steps, one reorder per step
    L, STEPS = 6, 150
    orders = [beam_order(g).to(d) for _ in range(STEPS)]
    xs = torch.randn(STEPS, 1, BSZ, D, device=d, generator=gd)

    def loop_ours(prec):
        layers = [make_module(prec) for _ in range(L)]
        inc = {}
        for s in range(STEPS):
            for m in layers:
                if s:
                    m.reorder_incremental_state(inc, orders[s])
                m(xs[s], None, None, incremental_state=inc, need_weights=False)

    def loop_torch():
        sts = [{} for _ in range(L)]
        for s in range(STEPS):
            for st in sts:
                torch_step(xs[s], st, orders[s] if s else None)

    for name, fn in (("DecoderSelfAttention bf16", lambda: loop_ours("bf16")),
                     ("DecoderSelfAttention fp32", lambda: loop_ours("fp32")),
                     ("torch restatement fp32", loop_torch)):
        fn()  # warm-up: allocator, module load
        ts = []
        for _ in range(3):
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e) / STEPS)
        print("decode loop %-27s %d layers x %d steps: %.3f ms/step (median of 3 loops; all: %s)" %
              (name, L, STEPS, sorted(ts)[1], " ".join("%.3f" % v for v in ts)), flush=True)
